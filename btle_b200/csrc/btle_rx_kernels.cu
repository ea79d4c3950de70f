// btle_rx_kernels.cu — sm_100a kernels of the BLE receive path + the C-ABI (include/btle_b200.h).
//
// btle_rx_persistent_kernel does the whole receive chain of the reference's receiver()
// (btle_rx.c:2188-2391): one persistent, warp-specialised CTA per SM.
//   dense warps     IQ tile (two TMA boxes, 128B swizzle) -> per-lane discriminator bits packed into
//                   phase words (btle_core.cuh: 1 PRMT + 2 IDP.2A + 1 SHF per sample) -> 12-tap
//                   bit-parallel prefilter of the 32-tap access-address match against the neighbour
//                   lane's words (__shfl_down_sync) -> candidate words + group flags (ballot)
//   resolver warps  one lane per chunk replays the reference's greedy loop on the phase words:
//                   zero-history partial windows, exact re-check of candidates, dewhiten, header
//                   parse, length guards, CRC-24 (4 bytes per step), 64-byte record appended
//   ring            4 span slots between them, mbarrier full/empty protocol
// Also here: leaf kernels with the reference's function signatures (unit parity), the Python
// model's receiver batched one warp per packet, and the transmit PHY (4- and 8-sps modulators).
// No tensor cores: the path has no dense contraction (integer compare / bit work on a stream).
#include <cuda.h>
#include <cuda_runtime.h>

#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/btle_b200.h"
#include "btle_core.cuh"
#include "btle_params.h"
#include "btle_wideband.h"

using namespace btle;

// ----------------------------------------------------------------------------------------------
// protocol tables in constant memory (generated at context creation, verified against the
// reference's scramble_table.h / crc_table in tests)
__constant__ uint32_t c_whiten_words[40][12];
__constant__ uint32_t c_crc4[1024];
__constant__ int8_t c_cos1024[1024], c_sin1024[1024];   // round(127 cos/sin(2 pi k/1024)), gauss_cos_sin_table.h
__constant__ int8_t c_cos2048[2048], c_sin2048[2048];   // btlelib.py:52-66 (sin_cos_gen)
__constant__ int c_gauss4[9] = {2, 11, 32, 53, 60, 53, 32, 11, 2};                       // btle_tx.c gauss_coef_int8[4..12]
__constant__ int c_gauss8[17] = {0, 0, 0, 1, 4, 9, 15, 22, 24, 22, 15, 9, 4, 1, 0, 0, 0};  // btlelib.py:146-160   // c_crc4[0..255] == crc_table (btle_rx.c:971-1004)

static_assert(sizeof(btle_pkt_rec) == 64, "record must be 64 bytes");
static_assert(sizeof(btle_stream_cfg) == 24, "cfg must be 24 bytes");
static_assert(sizeof(btle_model_rx_rec) == 80, "model rx record must be 80 bytes");
static_assert(sizeof(btle_synth_truth) == 64, "synth truth record must be 64 bytes");
static_assert(sizeof(btle_sps8_rec) == 96, "sps8 record must be 96 bytes");

#ifdef BTLE_TIMING
// diagnostic builds only (tools/diag_timing.py): per-CTA time stamps in ns
__device__ unsigned long long g_timing[148 * 16];
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define BTLE_STAMP(slot) do { if (lane == 0) atomicMax(&g_timing[(blockIdx.x % 148) * 16 + (slot)], gtime()); } while (0)
#define BTLE_STAMP_MIN(slot) do { if (lane == 0) atomicMin(&g_timing[(blockIdx.x % 148) * 16 + (slot)], gtime()); } while (0)
extern "C" void btle_b200_debug_timing(unsigned long long *dst, int reset) {
  if (reset) { static unsigned long long z[148 * 16]; for (int i = 0; i < 148 * 16; ++i) z[i] = (i % 16 == 0 || i % 16 == 2) ? ~0ull : 0ull; cudaMemcpyToSymbol(g_timing, z, sizeof z); }
  else cudaMemcpyFromSymbol(dst, g_timing, sizeof(unsigned long long) * 148 * 16);
}
#else
#define BTLE_STAMP(slot) do { } while (0)
#define BTLE_STAMP_MIN(slot) do { } while (0)
#endif

namespace {

// ---- launch shape -----------------------------------------------------------------------------
#ifndef BTLE_DENSE_WARPS
#define BTLE_DENSE_WARPS 16
#endif
#ifndef BTLE_RESOLVE_WARPS
#define BTLE_RESOLVE_WARPS 3
#endif
#ifndef BTLE_SLOTS
#define BTLE_SLOTS 4
#endif
#ifndef BTLE_CTAS_PER_SM
#define BTLE_CTAS_PER_SM 1     // (A/B builds: 2 CTAs of 7 dense + 2 resolver warps and 2 slots share one SM)
#endif
constexpr int kCtasPerSm = BTLE_CTAS_PER_SM;
constexpr int kDenseWarps = BTLE_DENSE_WARPS;  // producers: IQ -> phase words + candidate words
constexpr int kResolveWarps = BTLE_RESOLVE_WARPS;   // consumers: per-chunk greedy decode (alternate spans)
constexpr int kThreads = (kDenseWarps + kResolveWarps) * 32;
// kSpanChunks = 16 chunks per span (btle_core.cuh): one resolver lane per chunk in the chain pass
constexpr int kSlots = BTLE_SLOTS;             // ring of span buffers between producers and consumers
constexpr int kSpanGroups = kGroupsPerChunk * kSpanChunks + kHaloGroups;   // 1036
constexpr int kStageBytes = 8192;              // one warp tile (32 groups = 4096 samples), two 4 KB halves
constexpr int kHaloRows = kHaloGroups;         // rows of the last (look-ahead) tile of a span: always 12

struct Slot {
  uint4 pd[kSpanGroups + 1];                   // phase words (+1 zero group behind the data)
  uint32_t cand[kSpanGroups + 4];              // candidate word per group (prefilter, any phase)
  uint32_t flagw[2 * kSpanChunks + 2];         // bit l of word t: group 32t+l has candidates
  StreamParams sp;
};

constexpr int kHitCap = BTLE_MAX_PKTS_PER_CHUNK + kMaxRejectedPerChunk + 1;    // counted + reported-rejected hits per chunk (68 x u16)
struct ResolveScratch {                        // per resolver warp, between the chain pass and the decode pass
  uint16_t hit[kSpanChunks][kHitCap];          // n0 + 124 of every counted packet, per chunk, in the reference's order
  uint16_t pre[kSpanChunks + 2];               // exclusive prefix of the per-chunk counts; [kSpanChunks] = total
  uint16_t xh[2 * kSpanChunks][kExactCap + 1]; // exact access-address hits per flag word (offsets inside the word); [kExactCap] = count
};

struct Smem {
  Slot slot[kSlots];
  uint32_t crc4[1024];
  ResolveScratch rs[kResolveWarps];
  alignas(1024) unsigned char stage[kDenseWarps][kStageBytes];
  alignas(8) unsigned long long mbar[2 * kDenseWarps];   // TMA completion, two per dense warp
  unsigned long long full[kSlots];                        // kDenseWarps arrivals: span published
  unsigned long long empty[kSlots];                       // 1 arrival: span consumed
};

static_assert(sizeof(Smem) <= (kCtasPerSm == 1 ? 232448 : 116224 - 1024), "Smem exceeds what a CTA can have on sm_100");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// Ring barriers may stay closed for microseconds: poll politely so the spin does not eat issue slots.
__device__ __forceinline__ void mbar_wait_backoff(unsigned long long *bar, uint32_t parity) {
  uint32_t done = 0;
  for (;;) {
#ifdef BTLE_WAIT_HINT
    // suspend-time hint: the warp sleeps inside the barrier unit and is woken by the phase change, instead of polling
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity), "r"(4000u) : "memory");
    if (done) break;
    __nanosleep(500);
#else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (done) break;
    __nanosleep(200);
#endif
  }
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
  asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA tiled copy (cp.async.bulk.tensor, SASS UTMALDG): box {128 B, 1 half, rows, 1 stream} of the
// IQ tensor {128 B, 2 halves, 256-byte runs, streams} -> shared, 128B-swizzled, completion counted
// in bytes on an mbarrier.
__device__ __forceinline__ void tma_load_half(void *smem_dst, const CUtensorMap *map, int half, int run, int stream,
                                              unsigned long long *bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(0), "r"(half), "r"(run), "r"(stream), "r"(smem_u32(bar)) : "memory");
}
// Writes one packet record.  Reads the raw IQ only when the caller asked for RSSI.
__device__ __forceinline__ void store_record(btle_pkt_rec *dst, int stream, int chunk, int n0, int nbytes, int crc_bad, bool rejected,
                                             const uint32_t words[11], const StreamParams &sp, const int8_t *iq,
                                             long long n_int8, long long lead) {
  uint32_t mag = 0;
  if (sp.rssi) {                                            // btle_rx.c:2234-2243
    const long long first = (long long)chunk * kChunkInt8 + 2ll * n0;
    for (int k = 0; k < 256; ++k) {
      const long long a = first + k;
      int v = (a >= -lead && a < n_int8) ? (int)iq[a] : 0;     // `lead` bytes in front of the capture are readable (stream segments)
      mag += (uint32_t)(v < 0 ? -v : v);
    }
  }
  uint32_t r[16];
  r[0] = (uint32_t)stream;
  r[1] = (uint32_t)chunk;
  r[2] = (uint32_t)n0;
  r[3] = (uint32_t)sp.channel | ((uint32_t)nbytes << 8) | ((uint32_t)crc_bad << 16) |
         ((uint32_t)((sp.raw ? 1 : 0) | (sp.adv ? 2 : 0) | (rejected ? BTLE_REC_REJECTED : 0)) << 24);
  r[4] = sp.aa;
  r[5] = (mag & 0xFFFFu) | (words[0] << 16);                // mag_sum, bytes[0..1]
#pragma unroll
  for (int j = 1; j < 11; ++j) r[5 + j] = (words[j - 1] >> 16) | (words[j] << 16);
  uint4 *d4 = reinterpret_cast<uint4 *>(dst);
#pragma unroll
  for (int q = 0; q < 4; ++q) d4[q] = make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
}

// Copy one stream's parameters (built on the host by make_params(), uploaded next to the cfg array) into a ring slot:
// one coalesced load of sizeof(StreamParams) = 184 bytes by a warp, no dependent look-ups.
constexpr int kParamWords = (int)(sizeof(StreamParams) / 4);
static_assert(sizeof(StreamParams) % 4 == 0 && kParamWords <= 64, "StreamParams is copied as <= 2 words per lane");
__device__ __forceinline__ void load_params_warp(const StreamParams *__restrict__ src, StreamParams &dst, int lane) {
  const uint32_t *s = reinterpret_cast<const uint32_t *>(src);
  uint32_t *d = reinterpret_cast<uint32_t *>(&dst);
  const uint32_t a = __ldg(s + lane);
  uint32_t b = 0;
  if (lane + 32 < kParamWords) b = __ldg(s + lane + 32);
  d[lane] = a;
  if (lane + 32 < kParamWords) d[lane + 32] = b;
}

// One persistent CTA per SM.  Units of work (a span of 16 chunks of one capture, or a 4-chunk piece of one in the
// last wave — Plan, btle_core.cuh) are dealt round-robin to CTAs.
// Warps 0..15 (dense): per 4096-sample tile, two TMA boxes bring the tile into 128B-swizzled shared rows;
//   each lane turns its 128 samples into 4 phase words, prefilters the access-address match against
//   the neighbour lane's words (warp shuffle) and publishes both in the unit's ring slot.
// Warps 16..18 (resolvers, units k = r, r+3, ...): when a unit is complete,
//   1. chain pass, one lane per chunk: the reference's greedy receiver() control flow (search, header length,
//      guards) on the phase words -> positions of the packets the reference counts;
//   2. one warp scan + ONE atomic reserve the unit's block of the output and fill the unit's directory entry;
//   3. decode pass, one lane per PACKET (converged): bytes, dewhitening, CRC-24, 64-byte record stored at its
//      final position — records of a unit are contiguous and in the reference's order.
// Producers and consumers are decoupled through a 4-slot ring with full/empty mbarriers, so the sparse
// passes of unit k overlap the dense pass of units k+1 .. k+3.
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
btle_rx_persistent_kernel(const __grid_constant__ CUtensorMap map32, const __grid_constant__ CUtensorMap map12,
                          const int8_t *__restrict__ iq, long long stream_stride, long long n_int8,
                          const StreamParams *__restrict__ params, const Plan plan,
                          btle_pkt_rec *__restrict__ out, unsigned cap, unsigned *__restrict__ count,
                          uint2 *__restrict__ dir, unsigned *__restrict__ zero_next, long long lead) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem &M = *reinterpret_cast<Smem *>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int total_units = plan.total_units;

  BTLE_STAMP_MIN(0);
  // context-owned allocation counters rotate through a ring: this launch clears the one a launch half a ring later will use
  if (zero_next && blockIdx.x == 0 && tid == 0) *zero_next = 0u;
  // ---- dense warps: (span, tile) iterator and TMA request helpers -------------------------------------
  // Each warp walks its own sequence of tiles (tile j of the CTA goes to warp j % 16, across
  // unit boundaries).  A tile is fetched as two 4 KB TMA boxes — the upper and the lower 128
  // bytes of every lane's 256-byte run — each into its own buffer; as soon as a half has been
  // consumed the same half of the warp's NEXT tile is requested into that buffer, so the copy of
  // the next tile overlaps the arithmetic of this one.
  unsigned char *stage = M.stage[warp < kDenseWarps ? warp : 0];
  unsigned long long *mbar = &M.mbar[2 * (warp < kDenseWarps ? warp : 0)];   // [0] lower-half buffer, [1] upper-half buffer
  // How a tile's bytes get into shared memory.  The tensor map has n_int8/256 rows per capture; rows behind them read
  // as ZERO through TMA (out-of-bounds fill), which is exactly what the reference-equivalent semantics want for the
  // look-ahead behind the end of a capture.  Only a capture whose length is not a multiple of 256 has one partial row
  // that TMA would zero as a whole: the tile that holds it is filled by hand.  A tile entirely behind the capture
  // (the look-ahead tile of a capture's last span) is zeroed in place.
  const int runs = (int)(n_int8 >> 8);
  const bool ragged = (n_int8 & 255) != 0;
  auto tile_mode = [&](int run0, int rows) {              // 0 TMA, 1 by hand, 2 zeros
    if (run0 >= runs + (ragged ? 1 : 0)) return 2;
    return (ragged && runs < run0 + rows) ? 1 : 0;
  };
  struct Cursor {                                         // (unit, tile) iterator of this warp
    int unit, t, rot, tiles, groups, chunk0, stream;
    bool valid;
  };
  auto enter_unit = [&](Cursor &c) {
    c.valid = c.unit < total_units;
    if (c.valid) {
      const UnitInfo ui = unit_info(c.unit, plan);
      c.tiles = ui.tiles; c.groups = ui.groups; c.chunk0 = ui.chunk0; c.stream = ui.stream;
      c.t = warp - c.rot;
      if (c.t < 0) c.t += kDenseWarps;
    }
  };
  auto next_unit = [&](Cursor &c) {
    c.rot = (c.rot + c.tiles) % kDenseWarps;
    c.unit += gridDim.x;
    enter_unit(c);
  };
  auto next_tile = [&](Cursor &c) {                       // next tile of this warp, skipping empty units
    c.t += kDenseWarps;
    while (c.valid && c.t >= c.tiles) next_unit(c);
  };
  // descriptor of the tile under the prefetch cursor, refreshed once per tile
  int nx_run0 = 0, nx_stream = 0;
  uint32_t nx_bytes = 0;                                  // bytes per half; 0 = nothing to request by TMA
  const CUtensorMap *nx_map = &map32;
  auto describe = [&](const Cursor &c) {
    nx_bytes = 0;
    if (!c.valid) return;
    const int rows = min(32, c.groups - c.t * 32);
    nx_run0 = c.chunk0 * 64 + c.t * 32;
    nx_stream = c.stream;
    nx_map = (rows == 32) ? &map32 : &map12;
    if (tile_mode(nx_run0, rows) == 0) nx_bytes = (uint32_t)rows * 128u;   // else: filled by the consumer itself
  };
  auto request_half = [&](int half) {                     // 1 = upper, 0 = lower half of the described tile
    if (lane == 0 && nx_bytes) {
      mbar_expect_tx(&mbar[half], nx_bytes);
      tma_load_half(stage + (half << 12), nx_map, half, nx_run0, nx_stream, &mbar[half]);
    }
  };
  Cursor pf;                                              // the tile to request next
  pf.unit = blockIdx.x; pf.rot = 0; pf.valid = false; pf.t = 0; pf.tiles = 0; pf.groups = 0; pf.chunk0 = 0; pf.stream = 0;

  // Start-up.  Warps 0..3 fetch the parameters of the CTA's first four units; their loads are issued BEFORE the tile
  // requests (148 CTAs x 16 warps x 8 KB of TMA traffic would otherwise sit in front of them in the memory system)
  // and consumed after, so both round trips overlap.
  uint32_t pw0 = 0, pw1 = 0;
  const int first_unit = blockIdx.x + warp * gridDim.x;
  const bool has_params = warp < kSlots && first_unit < total_units;
  if (has_params) {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(params + unit_info(first_unit, plan).stream);
    pw0 = __ldg(src + lane);
    if (lane + 32 < kParamWords) pw1 = __ldg(src + lane + 32);
  }
  if (warp < kDenseWarps) {
    // the first tile is requested right away: its HBM round trip overlaps the rest of the start-up
    if (lane == 0) {
      mbar_init(&mbar[0], 1);
      mbar_init(&mbar[1], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    enter_unit(pf);
    while (pf.valid && pf.t >= pf.tiles) next_unit(pf);
    describe(pf);
    request_half(1);
    request_half(0);
    next_tile(pf);
    describe(pf);
    BTLE_STAMP(10);
  }
  if (tid < kSlots) { mbar_init(&M.full[tid], kDenseWarps); mbar_init(&M.empty[tid], 1); }
  if (has_params) {
    uint32_t *d = reinterpret_cast<uint32_t *>(&M.slot[warp].sp);
    d[lane] = pw0;
    if (lane + 32 < kParamWords) d[lane + 32] = pw1;
    BTLE_STAMP(11);
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  BTLE_STAMP(1);

  if (warp < kDenseWarps) {
    // =============================== dense producers ===============================
    uint32_t tma_phase = 0;                               // bit h: parity to wait for on buffer h
    int rot = 0, k = 0;
    for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x, ++k) {
      const int b = k % kSlots;
      Slot &S = M.slot[b];
      const uint32_t use = (uint32_t)(k / kSlots);
      if (use > 0) mbar_wait_backoff(&M.empty[b], (use - 1) & 1u);   // resolver released the slot's previous unit
      const UnitInfo si = unit_info(unit, plan);
      const int8_t *cap_base = iq + (long long)si.stream * stream_stride;
      int t = warp - rot;
      if (t < 0) t += kDenseWarps;
      for (; t < si.tiles; t += kDenseWarps) {
        const int rows = min(32, si.groups - t * 32);
        const int run0 = si.chunk0 * 64 + t * 32;
        const long long tile_off = (long long)run0 * 256;
        const int mode = tile_mode(run0, rows);
        const bool tma = mode == 0;
        // first IQ word behind the tile: the sample after the last row's run
        uint32_t tail = 0;
        if (lane == rows - 1) {
          const long long o = tile_off + (long long)rows * 256;
          if (o + 4 <= n_int8) tail = __ldg(reinterpret_cast<const uint32_t *>(cap_base + o));
          else
            for (int bb = 0; bb < 4; ++bb)
              if (o + bb < n_int8) tail |= (uint32_t)(uint8_t)cap_base[o + bb] << (8 * bb);
        }
        uint32_t acc[4] = {0u, 0u, 0u, 0u};
        uint32_t carry = 0u, wtop = 0u;
        int vtop = 0;
#pragma unroll 1
        for (int half = 1; half >= 0; --half) {
          unsigned char *buf = stage + (half << 12);
          if (tma) {
            mbar_wait(&mbar[half], (tma_phase >> half) & 1u);
            tma_phase ^= 1u << half;
          } else if (mode == 2) {
            if (lane < rows) {
#pragma unroll
              for (int cc = 0; cc < 8; ++cc) *reinterpret_cast<uint4 *>(buf + (lane << 7) + (cc << 4)) = make_uint4(0u, 0u, 0u, 0u);
            }
            __syncwarp();
          } else {
            // the capture's partial last row: bytes past n_int8 read as 0 (same swizzled layout, generic stores)
            if (lane < rows) {
              const long long row_off = tile_off + (long long)lane * 256 + 128 * half;
              for (int wi = 0; wi < 32; ++wi) {
                const long long o = row_off + 4ll * wi;
                uint32_t w = 0;
                if (o + 4 <= n_int8) w = *reinterpret_cast<const uint32_t *>(cap_base + o);
                else
                  for (int bb = 0; bb < 4; ++bb)
                    if (o + bb < n_int8) w |= (uint32_t)(uint8_t)cap_base[o + bb] << (8 * bb);
                reinterpret_cast<uint32_t *>(buf + (lane << 7) + ((((wi >> 2) ^ (lane & 7))) << 4))[wi & 3] = w;
              }
            }
            __syncwarp();
          }
          // 16-byte chunk cc of this lane's 128-byte row sits at cc ^ (lane & 7) (TMA SWIZZLE_128B):
          // the 8 lanes of a quarter-warp hit 8 different bank groups -> conflict-free LDS.128
          const unsigned char *row = buf + (lane << 7);
          const uint32_t sw = (uint32_t)(lane & 7);
          if (half == 0) {
            // now the neighbour's first word is here: redo the one bit that needed it (sample 127)
            const uint32_t first = reinterpret_cast<const uint4 *>(row + (sw << 4))->x;
            uint32_t nb = __shfl_down_sync(0xFFFFFFFFu, first, 1);
            if (lane == rows - 1) nb = tail;
            vtop = sext8<3>(wtop) * sext8<0>(nb) - sext8<2>(wtop) * sext8<1>(nb);
          }
          if (lane < rows) {
#pragma unroll
            for (int cc = 7; cc >= 0; --cc) {
              const uint4 w = *reinterpret_cast<const uint4 *>(row + ((((uint32_t)cc ^ sw)) << 4));
              if (half == 1 && cc == 7) wtop = w.w;
#ifdef BTLE_DBITS_PUSH
              dbits8(w.x, w.y, w.z, w.w, carry, acc);
#else
              if ((cc & 3) == 3) {                          // next byte of the phase words (the walk goes downwards)
#pragma unroll
                for (int ph = 0; ph < 4; ++ph) acc[ph] <<= 8;
              }
              switch (cc & 3) {
                case 3: dbits8_dense<3>(w.x, w.y, w.z, w.w, carry, acc); break;
                case 2: dbits8_dense<2>(w.x, w.y, w.z, w.w, carry, acc); break;
                case 1: dbits8_dense<1>(w.x, w.y, w.z, w.w, carry, acc); break;
                default: dbits8_dense<0>(w.x, w.y, w.z, w.w, carry, acc); break;
              }
#endif
              carry = w.x;
            }
            // sample 127 was pushed first, so after all 32 pushes it is bit 31 of phase 3
            if (half == 0) acc[3] = (acc[3] & 0x7FFFFFFFu) | ((uint32_t)vtop & 0x80000000u);
          }
          __syncwarp();                                   // everyone is done reading this buffer
          request_half(half);                             // same half of the warp's next tile
        }
        next_tile(pf);
        describe(pf);
        BTLE_STAMP_MIN(2);
        if (lane < rows) S.pd[t * 32 + lane] = make_uint4(acc[0], acc[1], acc[2], acc[3]);
        // candidate words: lanes 0..30 see the next group's words through the warp; lane 31 of
        // a full tile is completed by the resolver (its neighbour group belongs to another warp)
        uint32_t hi[4];
#pragma unroll
        for (int ph = 0; ph < 4; ++ph) hi[ph] = __shfl_down_sync(0xFFFFFFFFu, acc[ph], 1);
        uint32_t a = 0u;
        if (t < 2 * si.nch && lane < 31) a = prefilter_any(acc, hi, S.sp);
        const uint32_t fw = __ballot_sync(0xFFFFFFFFu, a != 0u);
        if (lane < rows) S.cand[t * 32 + lane] = a;
        if (lane == 0) {
          S.flagw[t] = fw;
          if (t == si.tiles - 1) S.pd[si.groups] = make_uint4(0u, 0u, 0u, 0u);
        }
      }
      rot = (rot + si.tiles) % kDenseWarps;
      __syncwarp();
      if (lane == 0) mbar_arrive(&M.full[b]);             // release: this warp's share of the unit is published
      BTLE_STAMP(3);
    }
  } else {
    // ================================== resolvers ==================================
    // the CRC tables are only needed here: built by the resolver warps while the first unit is in flight
    // (crc4[0..255] = crc_table, btle_rx.c:971-1004; [256k..] = the same followed by k zero bytes)
    {
      const int rt = tid - kDenseWarps * 32, rn = kResolveWarps * 32;
      for (int i = rt; i < 256; i += rn) M.crc4[i] = make_crc_entry((uint32_t)i);
      asm volatile("bar.sync 1, %0;" ::"r"(rn) : "memory");
      for (int kk = 1; kk < 4; ++kk) {
        for (int i = rt; i < 256; i += rn) { const uint32_t x = M.crc4[(kk - 1) * 256 + i]; M.crc4[kk * 256 + i] = M.crc4[x & 0xFFu] ^ (x >> 8); }
        asm volatile("bar.sync 1, %0;" ::"r"(rn) : "memory");
      }
    }
    // resolver warp r takes this CTA's units k = r, r + kResolveWarps, ...
    ResolveScratch &RS = M.rs[warp - kDenseWarps];
    int k = warp - kDenseWarps;
    for (int unit = blockIdx.x + k * gridDim.x; unit < total_units; unit += kResolveWarps * gridDim.x, k += kResolveWarps) {
      const int b = k % kSlots;
      Slot &S = M.slot[b];
      mbar_wait_backoff(&M.full[b], (uint32_t)(k / kSlots) & 1u);   // all tiles of the unit are published
      BTLE_STAMP(4);
      const UnitInfo si = unit_info(unit, plan);
      const int8_t *cap_base = iq + (long long)si.stream * stream_stride;
      for (int t = lane; t < 2 * si.nch; t += 32) {       // lane 31 of every full tile
        const int g = 32 * t + 31;
        const uint4 lo = S.pd[g], hi = S.pd[g + 1];
        const uint32_t l4[4] = {lo.x, lo.y, lo.z, lo.w}, h4[4] = {hi.x, hi.y, hi.z, hi.w};
        const uint32_t a = prefilter_any(l4, h4, S.sp);
        S.cand[g] = a;
        if (a) S.flagw[t] |= 0x80000000u;
      }
      __syncwarp();
      BTLE_STAMP(6);
      // 1a. exact access-address hits of the unit, all lanes (lane = flag word = 32 groups): the only data-dependent search
      for (int t = lane; t < 2 * si.nch; t += 32)
        RS.xh[t][kExactCap] = (uint16_t)enumerate_exact_hits(reinterpret_cast<const uint32_t *>(S.pd), S.cand, S.flagw[t], t, S.sp, RS.xh[t]);
      __syncwarp();
      // 1b. chain pass: which hits does the reference count?  (lane = chunk; walks the chunk's two hit lists)
      int mine = 0;
      if (lane < si.nch) {
        struct Note {
          uint16_t *row;
          __device__ __forceinline__ void operator()(int i, int n0, bool rej) { row[i] = (uint16_t)((n0 + 124) | (rej ? 0x8000 : 0)); }
        } note{RS.hit[lane]};
        const uint32_t *pdc = reinterpret_cast<const uint32_t *>(&S.pd[kGroupsPerChunk * lane]);
        const int c0 = RS.xh[2 * lane][kExactCap], c1 = RS.xh[2 * lane + 1][kExactCap];
        if (c0 > kExactCap || c1 > kExactCap)              // degenerate mask: too many matches to list, walk the candidates instead
          mine = chain_chunk(pdc, &S.cand[kGroupsPerChunk * lane], &S.flagw[2 * lane], S.sp, note);
        else
          mine = chain_chunk_lists(pdc, RS.xh[2 * lane], c0, RS.xh[2 * lane + 1], c1, S.sp, note);
      }
      BTLE_STAMP(7);
      // 2. the unit's block of the output: exclusive scan of the per-chunk counts, one atomic for the unit
      int incl = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += v; }
      const int total = __shfl_sync(0xFFFFFFFFu, incl, 31);
      if (lane <= kSpanChunks) RS.pre[lane] = (uint16_t)(incl - mine);   // lanes >= nch hold `total`
      unsigned my_base = 0;
      if (lane == 0) {
        if (total) my_base = atomicAdd(count, (unsigned)total);
        dir[unit] = make_uint2(my_base, (unsigned)total);
      }
      __syncwarp();
      BTLE_STAMP(8);
      // 3. decode pass: one lane per packet, all lanes on the same instruction stream.  The reservation's result is
      //    only needed when the records are stored, so the atomic's round trip to L2 overlaps the decode.
      for (int j0 = 0; j0 < total; j0 += 32) {
        const int j = j0 + lane;
        uint32_t words[11];
        int nbytes = 0, crc_bad = 0, n0 = 0, c = 0;
        bool rej = false;
        if (j < total) {
          // chunk of packet j: pre[c] <= j < pre[c + 1]
#pragma unroll
          for (int step = kSpanChunks / 2; step >= 1; step >>= 1)
            if ((int)RS.pre[c + step] <= j) c += step;
          const int h = (int)RS.hit[c][j - (int)RS.pre[c]];
          rej = (h & 0x8000) != 0;
          n0 = (h & 0x7FFF) - 124;
          decode_packet(reinterpret_cast<const uint32_t *>(&S.pd[kGroupsPerChunk * c]), S.sp, M.crc4, n0, rej, words, nbytes, crc_bad);
        }
        const unsigned base = __shfl_sync(0xFFFFFFFFu, my_base, 0);
        if (j < total && base + (unsigned)j < cap)
          store_record(out + base + j, si.stream, si.chunk0 + c, n0, nbytes, crc_bad, rej, words, S.sp, cap_base, n_int8, lead);
      }
      BTLE_STAMP(9);
      __syncwarp();
      // the slot is reused by unit k + kSlots of this CTA: refresh its parameters if the stream changes
      const int next = unit + kSlots * gridDim.x;
      if (next < total_units) {
        const int ns = unit_info(next, plan).stream;
        if (ns != si.stream) load_params_warp(params + ns, S.sp, lane);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&M.empty[b]);            // release the slot to the producers
      BTLE_STAMP(5);
    }
  }
}

// ---- leaf kernels (unit parity through the C-ABI; not performance paths) ------------------------
__global__ void dbits_kernel(const int8_t *iq, long long n_samples, uint8_t *d) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_samples) return;
  const int i0 = iq[2 * n], q0 = iq[2 * n + 1], i1 = iq[2 * n + 2], q1 = iq[2 * n + 3];
  d[n] = (uint8_t)((i0 * q1 - i1 * q0) > 0);            // btle_rx.c:1533
}

// search_unique_bits (btle_rx.c:1510): one CTA; phase words and candidate words for the searched
// range, then lane 0 runs search_from() with R = 0.  ngroups*128 samples must be readable (+1).
__global__ void search_kernel(const int8_t *iq, int search_len, btle_stream_cfg cfg, int ngroups, uint32_t *pd,
                              uint32_t *cand, int *result) {
  __shared__ StreamParams sp;
  __shared__ uint32_t flagw[8];
  if (threadIdx.x == 0) make_params(cfg, c_whiten_words[cfg.channel], sp);
  if (threadIdx.x < 8) flagw[threadIdx.x] = 0u;
  for (int g = threadIdx.x; g < ngroups + 1; g += blockDim.x) {
    uint32_t acc[4] = {0u, 0u, 0u, 0u};
    if (g < ngroups) {
      const uint32_t *w = reinterpret_cast<const uint32_t *>(iq) + 64 * (long long)g;
      uint32_t carry = w[64];
      for (int c = 15; c >= 0; --c) {
        dbits8(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3], carry, acc);
        carry = w[4 * c];
      }
    }
    for (int ph = 0; ph < 4; ++ph) pd[4 * g + ph] = acc[ph];
  }
  __syncthreads();
  for (int g = threadIdx.x; g < ngroups; g += blockDim.x) {
    const uint32_t a = prefilter_any(&pd[4 * g], &pd[4 * (g + 1)], sp);
    cand[g] = a;
    if (a) atomicOr(&flagw[g >> 5], 1u << (g & 31));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int n0 = 0;
    const bool hit = search_from(pd, cand, flagw, 0, 4 * search_len - 124, sp, ngroups + 1, ngroups - 1, n0);
    *result = hit ? 2 * n0 : -1;                          // return value, btle_rx.c:1550/:1561
  }
}

__global__ void demod_byte_kernel(const int8_t *rxp, int num_byte, uint8_t *out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= num_byte) return;
  uint32_t b = 0;
  for (int j = 0; j < 8; ++j) {                           // btle_rx.c:1496-1506
    const int8_t *p = rxp + 8 * (8 * k + j);
    b |= (uint32_t)(((int)p[0] * p[3] - (int)p[2] * p[1]) > 0) << j;
  }
  out[k] = (uint8_t)b;
}

__global__ void scramble_kernel(const uint8_t *in, int n, int channel, int off, uint8_t *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = off + i;
  out[i] = in[i] ^ (uint8_t)(c_whiten_words[channel][t >> 2] >> (8 * (t & 3)));   // btle_rx.c:1232-1237
}

__global__ void crc24_kernel(const uint8_t *in, int n, uint32_t init, uint32_t *out) {
  uint32_t crc = init & 0xFFFFFFu;
  for (int i = 0; i < n; ++i) crc = c_crc4[(crc ^ in[i]) & 0xFFu] ^ (crc >> 8);    // btle_rx.c:1215-1218
  *out = crc;
}

// stream_callback's sample reduction (btle_rx.c:307-308): int16 -> (x >> shift) & 0xFF
__global__ void iq16_to_iq8_kernel(const int16_t *__restrict__ in, long long n, int shift, int8_t *__restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = (int8_t)((in[i] >> shift) & 0xFF);
}

// ---- btlelib.py leaf kernels (python/btlelib.py) ------------------------------------------------
__global__ void gfsk_demod_i16_kernel(const int16_t *i, const int16_t *q, long long n, int8_t *bit, int32_t *sig) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k + 1 >= n) return;
  // int32 products with numpy's wrap-around semantics (btlelib.py:396)
  const uint32_t s = (uint32_t)((int32_t)i[k] * (int32_t)q[k + 1]) - (uint32_t)((int32_t)i[k + 1] * (int32_t)q[k]);
  sig[k] = (int32_t)s;
  bit[k] = (int8_t)((int32_t)s > 0);
}

__global__ void search_seq_kernel(const int8_t *bit, long long n, const int8_t *seq, int m, long long *first) {
  const long long s0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s0 + m > n) return;
  for (int j = 0; j < m; ++j)
    if (bit[s0 + j] != seq[j]) return;                    // btlelib.py:408
  atomicMin(reinterpret_cast<unsigned long long *>(first), (unsigned long long)s0);
}

// crc24_core, btlelib.py:191-219: 24-stage LFSR, feedback = stage 23 ^ input, taps into stages
// 0,1,3,4,6,9,10; the result is the register read from stage 23 down to 0.
__global__ void crc24_bits_kernel(const int8_t *in, long long n, const int8_t *init, int8_t *out) {
  uint32_t st = 0;                                         // bit k = stage k
  for (int k = 0; k < 24; ++k) st |= (uint32_t)(init[k] & 1) << k;
  for (long long t = 0; t < n; ++t) {
    const uint32_t fb = ((st >> 23) ^ (uint32_t)in[t]) & 1u;
    st = (st << 1) & 0xFFFFFFu;
    if (fb) st ^= 0x00065Bu;                               // stages 0,1,3,4,6,9,10
  }
  for (int k = 0; k < 24; ++k) out[k] = (int8_t)((st >> (23 - k)) & 1u);
}

// scramble_core, btlelib.py:226-263: same LFSR as scramble_table.h, applied bit by bit.
__global__ void scramble_bits_kernel(const int8_t *in, long long n, int channel, int8_t *out) {
  uint32_t reg = 1u;
  for (int i = 0; i < 6; ++i) reg |= ((uint32_t)(channel >> (5 - i)) & 1u) << (1 + i);
  for (long long t = 0; t < n; ++t) {
    const uint32_t o = (reg >> 6) & 1u;
    out[t] = (int8_t)((o + (uint32_t)in[t]) & 1u);
    reg = ((reg << 1) & 0x7Fu) | o;
    reg ^= o << 4;
  }
}

// Transmit PHY: one CTA per packet.  Every thread owns 8 consecutive output samples: frequency
// word per sample from the (at most 3 / 17) filter taps that see an impulse, block-wide inclusive
// scan for the phase, table lookup.  SPS == 4: btle_tx.c:1022-1063; SPS == 8: btlelib.py:146-189.
template <int SPS>
__global__ void __launch_bounds__(512)
tx_modulate_kernel(const uint8_t *__restrict__ air, const int32_t *__restrict__ nbytes, int max_bytes,
                   int8_t *__restrict__ out_i, int8_t *__restrict__ out_q) {
  __shared__ uint8_t sb[128];
  __shared__ int warp_tot[16];
  const int pkt = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = nbytes[pkt];
  for (int i = tid; i < 128; i += blockDim.x) sb[i] = (i < nb) ? air[(size_t)pkt * max_bytes + i] : 0;
  __syncthreads();
  const int nbit = 8 * nb;
  const int nsamp = nbit * SPS + 16, nsamp_max = 8 * max_bytes * SPS + 16;
  auto pm1 = [&](int k) { return ((sb[k >> 3] >> (k & 7)) & 1) ? 1 : -1; };
  int run = 0;                                             // phase carried through the whole packet
  for (int base = 0; base < nsamp_max; base += 8 * blockDim.x) {
    const int s0 = base + 8 * tid;
    int f[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int m = s0 + u;                                // frequency word whose running sum is the phase
      int acc = 0;
      if (SPS == 4) {
        // acc_m = sum_{j=3..11} g[15-j] * os[m+j], impulse of symbol k at os[15+4k] (btle_tx.c:1052-1056)
        if (m < nsamp - 1) {
#pragma unroll
          for (int j = 3; j <= 11; ++j) {
            const int idx = m + j - 15;
            if (idx >= 0 && (idx & 3) == 0 && (idx >> 2) < nbit) acc += c_gauss4[j - 3] * pm1(idx >> 2);
          }
        }
      } else {
        // y[m] = sum_j taps[j] * x[17 - j + m], x = 17 x (-1), then the NRZ waveform (btlelib.py:163-167)
        if (m < nsamp) {
          int y = 0;
#pragma unroll
          for (int j = 3; j <= 13; ++j) {                  // taps outside 3..13 are zero
            const int xi = 17 - j + m;
            int x = 0;
            if (xi < 17) x = -1; else if (xi - 17 < 8 * nbit) x = pm1((xi - 17) >> 3);
            y += c_gauss8[j] * x;
          }
          acc = y >> 1;                                    // btlelib.py:177
        }
      }
      f[u] = acc;
    }
    int loc = 0;
#pragma unroll
    for (int u = 0; u < 8; ++u) { loc += f[u]; f[u] = loc; }               // inclusive within the thread
    int incl = loc;                                        // inclusive scan of thread totals across the block
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if (lane >= d) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int woff = 0, tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { if (w < warp) woff += warp_tot[w]; tot += warp_tot[w]; }
    const int excl = run + woff + incl - loc;              // sum of all frequency words before this thread's first
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int m = s0 + u;
      if (m >= nsamp_max) break;
      if (SPS == 4) {
        // sample m uses the phase BEFORE frequency word m is added (sample[0] = table[0], btle_tx.c:1046-1061)
        const int ph = (excl + (u ? f[u - 1] : 0)) & 1023;
        const bool on = m < nsamp;
        out_i[((size_t)pkt * nsamp_max + m) * 2] = on ? c_cos1024[ph] : 0;
        out_i[((size_t)pkt * nsamp_max + m) * 2 + 1] = on ? c_sin1024[ph] : 0;
      } else {
        const int ph = (excl + f[u]) & 2047;               // cumsum includes the current word (btlelib.py:97)
        const bool on = m < nsamp;
        out_i[(size_t)pkt * nsamp_max + m] = on ? c_cos2048[ph] : 0;
        out_q[(size_t)pkt * nsamp_max + m] = on ? c_sin2048[ph] : 0;
      }
    }
    run += tot;
    __syncthreads();
  }
}

// ---- capture synthesiser (test / benchmark input, SURVEY.md §8d C2-C5): noise floor + one burst per slot, all on
// the device.  Counter-based randomness (a 64-bit mix of seed, stream, position), so every byte of every capture is
// a pure function of (seed, stream, index) and a slot can be regenerated on its own.
__constant__ uint32_t c_noise_thr[13];     // P(round(N(-0.3, 0.8)) <= v) * 2^32 for v = -7 .. 5
__device__ __forceinline__ uint64_t mix64(uint64_t x) {          // splitmix64 finaliser
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__device__ __forceinline__ uint64_t draw(uint64_t seed, uint64_t stream, uint64_t a, uint64_t k) {
  return mix64(mix64(seed ^ (stream * 0xD1B54A32D192ED03ull)) ^ (a * 0x9E3779B97F4A7C15ull) ^ (k << 56));
}
__device__ __forceinline__ int noise_floor_value(uint32_t u) {
  int v = -7;
#pragma unroll
  for (int k = 0; k < 13; ++k) v += (u >= c_noise_thr[k]);
  return v;
}
// kind 0: integer noise floor of the reference capture (sigma 0.8 LSB, mean -0.3, clipped to [-7, 6]);
// kind 1: full-scale uniform int8 (a hot interferer: discriminator bits are 50/50); kind 2: zeros
__global__ void synth_noise_kernel(int8_t *__restrict__ iq, long long stride, long long n_int8, int n_streams, uint64_t seed, int kind) {
  const long long per = (n_int8 + 15) >> 4;                 // 16-byte pieces per capture
  const long long total = per * n_streams;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long s = i / per, p = i - s * per;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if (kind == 0) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const uint64_t r = draw(seed, (uint64_t)s, (uint64_t)p * 8 + q, 1);
        const uint32_t b0 = (uint32_t)noise_floor_value((uint32_t)r) & 0xFFu, b1 = (uint32_t)noise_floor_value((uint32_t)(r >> 32)) & 0xFFu;
        w[q >> 1] |= (b0 | (b1 << 8)) << (16 * (q & 1));
      }
    } else if (kind == 1) {
      const uint64_t r0 = draw(seed, (uint64_t)s, (uint64_t)p * 2, 1), r1 = draw(seed, (uint64_t)s, (uint64_t)p * 2 + 1, 1);
      w[0] = (uint32_t)r0; w[1] = (uint32_t)(r0 >> 32); w[2] = (uint32_t)r1; w[3] = (uint32_t)(r1 >> 32);
    }
    int8_t *dst = iq + s * stride + 16 * p;
    if (16 * p + 16 <= n_int8 && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) *reinterpret_cast<uint4 *>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
    else
      for (int b = 0; b < 16; ++b)
        if (16 * p + b < n_int8) dst[b] = (int8_t)(w[b >> 2] >> (8 * (b & 3)));
  }
}

struct SynthSlot { long long start; int n_air, pdu_len, corrupt_bit, straddle; };
// Placement and length of the burst of (stream, slot): needs only hashes, so a slot can ask about its predecessor.
__device__ SynthSlot synth_slot_geometry(const btle_synth_cfg &sc, const btle_stream_cfg &cfg, int stream, long long slot, long long n_samples,
                                         bool look_back) {
  SynthSlot g;
  const bool adv = cfg.channel >= 37;
  const uint64_t r = draw(sc.seed, (uint64_t)stream, (uint64_t)slot, 2);
  g.pdu_len = adv ? 2 + 6 + (int)(r % 32) : 2 + (int)(r % 28);               // ADV_IND: AdvA + 0..31 B; LL data: 0..27 B
  g.n_air = 1 + 4 + g.pdu_len + 3;
  const int n_s = 32 * g.n_air + 16;
  g.corrupt_bit = -1;
  if (sc.corrupt_every > 0 && slot % sc.corrupt_every == sc.corrupt_every - 1)
    g.corrupt_bit = g.pdu_len > 2 ? 16 + (int)((r >> 16) % (uint64_t)(8 * g.pdu_len - 16)) : 8 * g.pdu_len + 3;
  const long long S = sc.slot_samples;
  long long lo = slot * S;
  if (look_back && slot > 0 && sc.straddle_every > 0) {                       // a straddling predecessor spills into this slot
    const SynthSlot pv = synth_slot_geometry(sc, cfg, stream, slot - 1, n_samples, false);
    if (pv.straddle && pv.start + 32 * pv.n_air + 16 + 32 > lo) lo = pv.start + 32 * pv.n_air + 16 + 32;
  }
  long long hi = (slot + 1) * S - n_s;                                        // last start that keeps the burst in its slot
  if (hi < lo) hi = lo;
  g.start = lo + (long long)((r >> 32) % (uint64_t)(hi - lo + 1));
  g.straddle = 0;
  if (sc.straddle_every > 0 && slot % sc.straddle_every == sc.straddle_every - 1) {
    const long long edge = (slot * S / kChunkSamples + 1) * (long long)kChunkSamples;   // next chunk boundary behind the slot start
    const long long first = max(slot * S, edge - n_s + 1);
    if (first < edge && edge <= (slot + 1) * S && edge + n_s < n_samples) {
      g.start = first + (long long)((r >> 40) % (uint64_t)(edge - first));      // the boundary falls strictly inside the burst
      g.straddle = 1;
    }
  }
  return g;
}

// One CTA per (stream, slot): PDU from hashes -> CRC-24 -> whitening -> the btle_tx PHY (same arithmetic as
// tx_modulate_kernel<4>, btle_tx.c:1022-1063) -> scaled by amplitude/127 (floor) and added to the floor with saturation.
__global__ void __launch_bounds__(256)
synth_bursts_kernel(int8_t *__restrict__ iq, long long stride, long long n_int8, const btle_stream_cfg *__restrict__ cfgs,
                    const btle_synth_cfg sc, long long n_slots, btle_synth_truth *__restrict__ truth) {
  __shared__ uint8_t sb[64];
  __shared__ int warp_tot[8];
  __shared__ SynthSlot G;
  const long long gid = blockIdx.x;
  const int stream = (int)(gid / n_slots);
  const long long slot = gid - (long long)stream * n_slots;
  const btle_stream_cfg cfg = cfgs[stream];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long n_samples = n_int8 / 2;
  if (tid == 0) {
    G = synth_slot_geometry(sc, cfg, stream, slot, n_samples, true);
    const bool adv = cfg.channel >= 37;
    uint8_t pdu[48];
    const int plen = G.pdu_len - 2;
    if (adv) {
      pdu[0] = 0x40; pdu[1] = (uint8_t)plen;                                  // ADV_IND, TxAdd = 1
      const uint64_t adva = (uint64_t)slot | ((uint64_t)(stream & 0xFFFF) << 32);
      for (int b = 0; b < 6; ++b) pdu[2 + b] = (uint8_t)(adva >> (8 * b));
      for (int b = 6; b < plen; ++b) pdu[2 + b] = (uint8_t)(draw(sc.seed, (uint64_t)stream, (uint64_t)slot, 3 + (b >> 3)) >> (8 * (b & 7)));
    } else {
      const uint64_t r = draw(sc.seed, (uint64_t)stream, (uint64_t)slot, 2);
      pdu[0] = (uint8_t)((1 + ((r >> 8) & 1)) | ((slot & 1) << 2) | (((slot >> 1) & 1) << 3));   // LLID 1/2, NESN, SN
      pdu[1] = (uint8_t)plen;
      for (int b = 0; b < plen; ++b) pdu[2 + b] = (uint8_t)(draw(sc.seed, (uint64_t)stream, (uint64_t)slot, 3 + (b >> 3)) >> (8 * (b & 7)));
    }
    uint32_t crc = crc_init_reorder(cfg.crc_init);
    for (int b = 0; b < G.pdu_len; ++b) crc = c_crc4[(crc ^ pdu[b]) & 0xFFu] ^ (crc >> 8);
    uint8_t body[48];
    for (int b = 0; b < G.pdu_len; ++b) body[b] = pdu[b];
    body[G.pdu_len] = (uint8_t)crc; body[G.pdu_len + 1] = (uint8_t)(crc >> 8); body[G.pdu_len + 2] = (uint8_t)(crc >> 16);
    if (G.corrupt_bit >= 0) body[G.corrupt_bit >> 3] ^= (uint8_t)(1u << (G.corrupt_bit & 7));
    sb[0] = (cfg.access_addr & 1u) ? 0x55 : 0xAA;
    for (int b = 0; b < 4; ++b) sb[1 + b] = (uint8_t)(cfg.access_addr >> (8 * b));
    for (int b = 0; b < G.pdu_len + 3; ++b) sb[5 + b] = body[b] ^ (uint8_t)(c_whiten_words[cfg.channel][b >> 2] >> (8 * (b & 3)));
    for (int b = G.n_air; b < 64; ++b) sb[b] = 0;
    if (truth) {
      btle_synth_truth t;
      memset(&t, 0, sizeof t);
      t.start_sample = G.start; t.stream = stream; t.slot = (int32_t)slot;
      t.n_air_bytes = (uint8_t)G.n_air; t.corrupt = (uint8_t)(G.corrupt_bit >= 0); t.straddle = (uint8_t)G.straddle; t.pdu_len = (uint8_t)G.pdu_len;
      for (int b = 0; b < G.pdu_len; ++b) t.pdu[b] = pdu[b];
      truth[gid] = t;
    }
  }
  __syncthreads();
  const int nbit = 8 * G.n_air, nsamp = 4 * nbit + 16;
  auto pm1 = [&](int k) { return ((sb[k >> 3] >> (k & 7)) & 1) ? 1 : -1; };
  int8_t *cap_base = iq + (long long)stream * stride;
  // 8 samples per thread, 256 threads: 2048 >= 1520 samples, one pass
  const int s0 = 8 * tid;
  int f[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int m = s0 + u;
    int acc = 0;
    if (m < nsamp - 1) {
#pragma unroll
      for (int j = 3; j <= 11; ++j) {
        const int idx = m + j - 15;
        if (idx >= 0 && (idx & 3) == 0 && (idx >> 2) < nbit) acc += c_gauss4[j - 3] * pm1(idx >> 2);
      }
    }
    f[u] = acc;
  }
  int loc = 0;
#pragma unroll
  for (int u = 0; u < 8; ++u) { loc += f[u]; f[u] = loc; }
  int incl = loc;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += v; }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  int woff = 0;
  for (int w = 0; w < warp; ++w) woff += warp_tot[w];
  const int excl = woff + incl - loc;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int m = s0 + u;
    if (m >= nsamp) break;
    const int ph = (excl + (u ? f[u - 1] : 0)) & 1023;
    const long long a = 2 * (G.start + m);
    if (a + 1 >= n_int8) break;
    auto addsat = [&](long long at, int wave) {
      const int p = wave * sc.amplitude;
      const int scaled = p >= 0 ? p / 127 : -((-p + 126) / 127);              // floor division, like the numpy generator
      int v = (int)cap_base[at] + scaled;
      v = v > 127 ? 127 : (v < -128 ? -128 : v);
      cap_base[at] = (int8_t)v;
    };
    addsat(a, c_cos1024[ph]);
    addsat(a + 1, c_sin1024[ph]);
  }
}

// ---- 8 samples per symbol, streaming (SURVEY.md 8f-3): where does the access address occur, on which sample phase? ----
// Phase ph of an 8-Msps capture is the symbol-rate stream n = 8 s + ph; its bits are the Python model's
// gfsk_demodulation_fixed_point on samples 8 symbols apart (btlelib.py:395-400).  One CTA = 32 groups of 32 symbols
// (8192 samples, 32 KB of int16 IQ) + 8 samples of the next group:
//   load     the tile goes to shared memory with coalesced 16-byte loads (4 samples each), all of a thread's loads in
//            flight at once; a group's 256 sample words are stored 264 words apart, so that the compute phase — whose
//            warp reads 8 consecutive phases of 4 groups — touches 32 different banks
//   pack     thread (g, ph) packs the 32 bits of group g on phase ph into a word
//   match    and compares the 32 windows starting in its word against the access address (funnel shift with the next
//            group's word of the same phase)
constexpr int kSps8Groups = 32;
constexpr int kSps8Pitch = 264;                                             // words per group row in shared memory
constexpr int kSps8TileWords = (kSps8Groups + 1) * kSps8Pitch;
constexpr int kSps8Vec = (kSps8Groups + 1) * 64;                            // 16-byte vectors per tile (33 rows x 256 samples)
#ifndef BTLE_SPS8_BUFS
#define BTLE_SPS8_BUFS 1   // 1: one tile per CTA, 6 CTAs per SM hide each other's load phase (measured faster: 0.27 ms / GiB);
#endif                     // 2: persistent CTAs, next tile in flight while the current one is packed (0.32 ms: half the warps per SM)
constexpr int kSps8Bufs = BTLE_SPS8_BUFS;
constexpr size_t kSps8Smem = (kSps8Bufs * kSps8TileWords + (kSps8Groups + 1) * 8) * sizeof(uint32_t);   // tile buffer(s) + the bit words
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
// Tiles are copied global -> shared with cp.async (SASS LDGSTS).  The kernel body is written as a loop over tiles with
// kSps8Bufs buffers; the shipped configuration is one buffer and one tile per CTA (see BTLE_SPS8_BUFS).
__global__ void __launch_bounds__(256)
sps8_hits_kernel(const int16_t *__restrict__ iq, long long n_samples, long long n_tiles, uint32_t aa, long long *__restrict__ hits, unsigned cap,
                 unsigned *__restrict__ count) {
  extern __shared__ __align__(16) uint32_t sps8_smem[];
  // one word = (I, Q) of one sample.  (Buffer addresses are computed, not kept in an array: an indexed array of pointers
  // ends up in local memory and the tile accesses become generic loads instead of LDS.)
  auto tile_buf = [&](int b) -> uint32_t * { return sps8_smem + (kSps8Bufs > 1 ? b : 0) * kSps8TileWords; };
  uint32_t(*W)[8] = reinterpret_cast<uint32_t(*)[8]>(sps8_smem + kSps8Bufs * kSps8TileWords);
  const uint32_t *s32 = reinterpret_cast<const uint32_t *>(iq);
  const uint4 *s128 = reinterpret_cast<const uint4 *>(iq);                 // iq is 16-byte aligned
  // tile = 32 groups x 256 samples + the first 256 samples of the next group (only its first 8 are used, for bit 31 of the
  // last group; the full row keeps the copy regular)
  // a tile whose 33 staged rows and the one sample behind them lie inside the capture needs no range checks at all
  auto interior = [&](long long tile) { return (tile + 1) * (kSps8Groups * 256ll) + 256 + 8 <= n_samples; };
  auto issue = [&](uint32_t *T, long long tile) {
    const long long base = tile * (kSps8Groups * 256ll);
    if (interior(tile)) {
      const uint4 *src = s128 + base / 4 + threadIdx.x;
      uint32_t *dst = &T[(threadIdx.x >> 6) * kSps8Pitch + 4 * (threadIdx.x & 63)];
#pragma unroll
      for (int r = 0; r < 8; ++r) cp_async16(dst + r * 4 * kSps8Pitch, src + 256 * r);      // 256 vectors = 4 rows per step
      if (threadIdx.x < kSps8Vec - 2048) cp_async16(dst + 8 * 4 * kSps8Pitch, src + 2048);
    } else {
#pragma unroll 1
      for (int r = 0; r < 9; ++r) {
        const int k = threadIdx.x + 256 * r;
        if (k < kSps8Vec) {
          uint32_t *dst = &T[(k >> 6) * kSps8Pitch + 4 * (k & 63)];
          const long long n = base + 4ll * k;
          if (n + 4 <= n_samples) cp_async16(dst, s128 + base / 4 + k);
          else {                                                            // behind the capture / its last, partial vector
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            for (int q = 0; q < 4; ++q) if (n + q < n_samples) w[q] = __ldg(s32 + n + q);
            *reinterpret_cast<uint4 *>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  const int ph = threadIdx.x & 7, gl = threadIdx.x >> 3;
  int buf = 0;
  long long tile = blockIdx.x;
  if (tile < n_tiles) issue(tile_buf(0), tile);
  for (; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
    const long long next = tile + gridDim.x;
    if (kSps8Bufs > 1 && next < n_tiles) {
      issue(tile_buf(buf ^ 1), next);
      asm volatile("cp.async.wait_group 1;" ::: "memory");                 // the current tile has landed, the next may still fly
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const uint32_t *T = tile_buf(buf);
    const long long g0 = tile * kSps8Groups;
    auto bit = [](uint32_t cur, uint32_t nxt) -> uint32_t {
      const int i0 = (int16_t)(cur & 0xFFFF), q0 = (int16_t)(cur >> 16), i1 = (int16_t)(nxt & 0xFFFF), q1 = (int16_t)(nxt >> 16);
      // btlelib.py:396 computes i0*q1 - i1*q0 in int32; for int16 inputs the difference cannot wrap (|products| <= 2^30),
      // so its sign is the comparison of the two products
      return (uint32_t)(i0 * q1 > i1 * q0);
    };
    const bool inside = interior(tile);
    for (int gg = gl; gg <= kSps8Groups; gg += 32) {
      const long long n0 = (g0 + gg) * 256 + ph;
      const uint32_t *row = &T[gg * kSps8Pitch + ph];
      uint32_t w = 0, cur = row[0];
      if (gg < kSps8Groups) {
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const uint32_t nxt = (k < 31) ? row[8 * (k + 1)] : T[(gg + 1) * kSps8Pitch + ph];
          w |= bit(cur, nxt) << k;
          cur = nxt;
        }
      } else {
        // the look-ahead group's word (needed by windows that start in the tile's last group): 32 of its samples are in the
        // staged 33rd row, the last one belongs to the group behind it (L2: the next tile)
        const uint32_t behind = (n0 + 256 < n_samples) ? __ldg(s32 + n0 + 256) : 0u;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const uint32_t nxt = (k < 31) ? row[8 * (k + 1)] : behind;
          w |= bit(cur, nxt) << k;
          cur = nxt;
        }
      }
      if (!inside) {                                                        // bit k needs samples n0 + 8k and n0 + 8(k+1) inside the capture
        const long long room = (n_samples - 1 - n0) / 8;
        if (room < 32) w = room <= 0 ? 0u : (w & ((1u << room) - 1u));
      }
      W[gg][ph] = w;
    }
    __syncthreads();
    const uint32_t lo = W[gl][ph], hi = W[gl + 1][ph];
    // all 32 window starts at once: bit i of m survives if the window starting at bit i agrees with the access address on 8
    // of its 32 bits (every 4th), then the few survivors are compared exactly
    uint32_t m = 0xFFFFFFFFu;
#pragma unroll
    for (int p = 0; p < 32; p += 4) {
      const uint32_t f = funnel_r(lo, hi, (uint32_t)p);                     // bit i = stream bit i + p
      m &= ((aa >> p) & 1u) ? f : ~f;
    }
    while (m) {
      const int i = __ffs((int)m) - 1;
      m &= m - 1;
      if (funnel_r(lo, hi, (uint32_t)i) == aa) {
        const long long n = (g0 + gl) * 256 + 8ll * i + ph;                // first sample of the access address
        if (n + 8ll * 32 < n_samples) {                                    // all 32 bits lie inside the capture
          const unsigned k = atomicAdd(count, 1u);
          if (k < cap) hits[k] = n;
        }
      }
    }
    __syncthreads();                                                        // W and the consumed buffer are free again
    if (kSps8Bufs == 1 && next < n_tiles) issue(tile_buf(0), next);
  }
}

// ---- BER flow of python/test_btle_ber.py on the device: packet source + channel + int16 truncation --------------------
// One CTA per packet: 37 random payload bytes behind the fixed header 42 25 (test_btle_ber.py:27,:49), CRC-24, whitening,
// the Python model's 8-sps modulator (same arithmetic as tx_modulate_kernel<8>), add_freq_sampling_error (linear
// resampling at 1 + ppm/1e6 and the matching carrier rotation at 2450 MHz, btlelib.py:823-857), add_noise (AWGN,
// sigma = 127 / 10^(snr/20) / sqrt 2 per rail, :859-871), np.int16() truncation.  Counter-based randomness.
constexpr int kBerPduBytes = 39, kBerAirBytes = 1 + 4 + kBerPduBytes + 3, kBerSamples = 8 * 8 * kBerAirBytes + 16;   // 3024
__device__ __forceinline__ float2 gauss_pair(uint64_t r) {                 // Box-Muller on two 32-bit uniforms
  const float u1 = ((float)(uint32_t)r + 0.5f) * 2.3283064365386963e-10f;    // (0, 1)
  const float u2 = (float)(uint32_t)(r >> 32) * 2.3283064365386963e-10f;
  const float rad = sqrtf(-2.0f * __logf(u1));
  float sn, cs;
  sincospif(2.0f * u2, &sn, &cs);
  return make_float2(rad * cs, rad * sn);
}
__global__ void __launch_bounds__(384)
ber_synth_kernel(const btle_ber_cfg cfg, unsigned long long first_packet, int n_packets, int16_t *__restrict__ out_i, int16_t *__restrict__ out_q,
                 uint8_t *__restrict__ truth /*[n][40]*/) {
  __shared__ uint8_t sb[64];
  __shared__ int warp_tot[12];
  __shared__ float txi[kBerSamples + 8], txq[kBerSamples + 8];
  const int pkt = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (pkt >= n_packets) return;
  const unsigned long long gp = first_packet + (unsigned long long)pkt;
  if (tid == 0) {
    uint8_t pdu[kBerPduBytes];
    pdu[0] = 0x42; pdu[1] = 0x25;
    for (int b = 2; b < kBerPduBytes; ++b) pdu[b] = (uint8_t)(draw(cfg.seed, gp, (uint64_t)(b >> 3), 9) >> (8 * (b & 7)));
    uint32_t crc = crc_init_reorder(cfg.crc_init);
    for (int b = 0; b < kBerPduBytes; ++b) crc = c_crc4[(crc ^ pdu[b]) & 0xFFu] ^ (crc >> 8);
    sb[0] = (cfg.access_addr & 1u) ? 0x55 : 0xAA;
    for (int b = 0; b < 4; ++b) sb[1 + b] = (uint8_t)(cfg.access_addr >> (8 * b));
    for (int b = 0; b < kBerPduBytes + 3; ++b) {
      const uint8_t v = b < kBerPduBytes ? pdu[b] : (uint8_t)(crc >> (8 * (b - kBerPduBytes)));
      sb[5 + b] = v ^ (uint8_t)(c_whiten_words[cfg.channel][b >> 2] >> (8 * (b & 3)));
    }
    for (int b = kBerAirBytes; b < 64; ++b) sb[b] = 0;
    for (int b = 0; b < kBerPduBytes; ++b) truth[(size_t)pkt * 40 + b] = pdu[b];
  }
  __syncthreads();
  const int nbit = 8 * kBerAirBytes;
  auto pm1 = [&](int k) { return ((sb[k >> 3] >> (k & 7)) & 1) ? 1 : -1; };
  const int s0 = 8 * tid;
  int f[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int m = s0 + u;
    int acc = 0;
    if (m < kBerSamples) {
      int y = 0;
#pragma unroll
      for (int j = 3; j <= 13; ++j) {
        const int xi = 17 - j + m;
        int x = 0;
        if (xi < 17) x = -1; else if (xi - 17 < 8 * nbit) x = pm1((xi - 17) >> 3);
        y += c_gauss8[j] * x;
      }
      acc = y >> 1;
    }
    f[u] = acc;
  }
  int loc = 0;
#pragma unroll
  for (int u = 0; u < 8; ++u) { loc += f[u]; f[u] = loc; }
  int incl = loc;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += v; }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  int woff = 0;
  for (int w = 0; w < warp; ++w) woff += warp_tot[w];
  const int excl = woff + incl - loc;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int m = s0 + u;
    if (m < kBerSamples) {
      const int ph = (excl + f[u]) & 2047;
      txi[m] = (float)c_cos2048[ph];
      txq[m] = (float)c_sin2048[ph];
    }
  }
  __syncthreads();
  const double e = (double)cfg.ppm * 1e-6;
  const float sigma = 127.0f / exp10f(cfg.snr_db / 20.0f) * 0.70710678f;
  // carrier offset fo = e * 2450e6 Hz at the new sampling time (1/8 us) * (1 + e): cycles per sample
  const double cyc = e * 2450e6 * (0.125e-6 * (1.0 + e));
  for (int m = tid; m < kBerSamples; m += blockDim.x) {
    float vi = txi[m], vq = txq[m];
    if (cfg.ppm != 0.0f) {
      const double x = (double)m * (1.0 + e);                // np.interp(x, xp, i): linear, clamped to the last sample
      int k = (int)x;
      if (k >= kBerSamples - 1) { vi = txi[kBerSamples - 1]; vq = txq[kBerSamples - 1]; }
      else {
        const float fr = (float)(x - (double)k);
        vi = txi[k] + (txi[k + 1] - txi[k]) * fr;
        vq = txq[k] + (txq[k + 1] - txq[k]) * fr;
      }
      double turns = cyc * (double)m;
      turns -= floor(turns);
      float sn, cs;
      sincospif(2.0f * (float)turns, &sn, &cs);
      const float ri = vi * cs - vq * sn, rq = vi * sn + vq * cs;
      vi = ri; vq = rq;
    }
    const float2 g = gauss_pair(draw(cfg.seed, gp, (uint64_t)m, 10));
    out_i[(size_t)pkt * kBerSamples + m] = (int16_t)(vi + sigma * g.x);     // np.int16(): truncation toward zero
    out_q[(size_t)pkt * kBerSamples + m] = (int16_t)(vq + sigma * g.y);
  }
}

// test_btle_ber.py:62-72: bit errors are counted only in packets whose CRC failed; an empty rx_pdu_bit counts all 312 bits
__global__ void ber_score_kernel(const btle_model_rx_rec *__restrict__ rec, const uint8_t *__restrict__ truth, int n,
                                 unsigned long long *__restrict__ acc /*pkt_err, bit_err, aa_miss*/) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned err = 0, perr = 0, miss = 0;
  if (p < n) {
    const btle_model_rx_rec &r = rec[p];
    if (!r.crc_ok) {
      perr = 1;
      miss = r.found ? 0u : 1u;
      const int nb = r.n_pdu_bits;
      if (nb == 0) err = 8 * kBerPduBytes;
      else {
        const int common = min(nb, 8 * kBerPduBytes);
        for (int b = 0; b < (common + 7) / 8; ++b) {
          uint32_t d = (uint32_t)(r.pdu[b] ^ truth[(size_t)p * 40 + b]);
          const int rem = common - 8 * b;
          if (rem < 8) d &= (1u << rem) - 1u;
          err += __popc(d);
        }
      }
    }
  }
  // warp-level reduction, one atomic per warp and counter
  for (int d = 16; d; d >>= 1) { err += __shfl_down_sync(0xFFFFFFFFu, err, d); perr += __shfl_down_sync(0xFFFFFFFFu, perr, d); miss += __shfl_down_sync(0xFFFFFFFFu, miss, d); }
  if ((threadIdx.x & 31) == 0) {
    if (perr) atomicAdd(&acc[0], (unsigned long long)perr);
    if (err) atomicAdd(&acc[1], (unsigned long long)err);
    if (miss) atomicAdd(&acc[2], (unsigned long long)miss);
  }
}

// btlelib.btle_rx for a batch of packet windows: one warp per packet (see include/btle_b200.h).
constexpr int kModelMaxWords = 64;                         // <= 2048 symbols per window
// Sample a of packet p sits at g{i,q}[(base(p) + a) * elem_stride], base(p) = win_off ? win_off[p] : p * n_samples:
// a planar batch (elem_stride 1) or windows cut out of one interleaved int16 capture (gi = iq, gq = iq + 1, elem_stride 2).
__global__ void __launch_bounds__(128)
model_rx_batch_kernel(const int16_t *__restrict__ gi, const int16_t *__restrict__ gq, long long elem_stride,
                      const long long *__restrict__ win_off, int n_packets, int n_samples, int sps,
                      int adv, int channel, uint32_t aa, uint32_t crc_init, btle_model_rx_rec *__restrict__ out) {
  __shared__ uint32_t wh[26];                              // whitening stream, 800 bits (+pad)
  __shared__ uint32_t crc_tab[256];
  __shared__ uint32_t bw[4][kModelMaxWords + 2];           // demodulated bits of the current phase
  __shared__ uint32_t pw[4][20];                           // pdu words of the last phase that found the AA
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_tab[i] = c_crc4[i];
  if (threadIdx.x == 0) {                                  // scramble_core's LFSR (btlelib.py:226-263)
    uint32_t reg = 1u;
    for (int i = 0; i < 6; ++i) reg |= ((uint32_t)(channel >> (5 - i)) & 1u) << (1 + i);
    for (int w = 0; w < 26; ++w) {
      uint32_t v = 0;
      for (int b = 0; b < 32; ++b) {
        const uint32_t o = (reg >> 6) & 1u;
        v |= o << b;
        reg = ((reg << 1) & 0x7Fu) | o;
        reg ^= o << 4;
      }
      wh[w] = v;
    }
  }
  __syncthreads();
  const int pkt = blockIdx.x * 4 + warp;
  if (pkt >= n_packets) return;
  const long long base = win_off ? win_off[pkt] : (long long)pkt * n_samples;
  const int16_t *pi = gi + base * elem_stride, *pq = gq + base * elem_stride;
  const long long es = elem_stride;
  const int num_bit = n_samples / sps - 1;                 // btlelib.py:444 (n_samples % sps == 0)
  const int nw = (num_bit + 31) >> 5;
  uint32_t *B = bw[warp], *P = pw[warp];
  auto sbits = [&](int p) {                                // 32 stream bits from position p (p >= 0)
    return funnel_r(B[p >> 5], B[(p >> 5) + 1], (uint32_t)(p & 31));
  };
  auto wbits = [&](int p) { return funnel_r(wh[p >> 5], wh[(p >> 5) + 1], (uint32_t)(p & 31)); };
  int r_start = -1, r_plen = 0, r_npdu = 0, r_ok = 0, r_found = 0, r_phase = sps - 1;
  for (int w = lane; w < 20; w += 32) P[w] = 0u;
  for (int ph = 0; ph < sps; ++ph) {
    // gfsk_demodulation_fixed_point on i[ph::sps], q[ph::sps] (btlelib.py:395-400,461)
    for (int j = 0; j < nw; ++j) {
      const int k = 32 * j + lane;
      bool bit = false;
      if (k < num_bit) {
        const long long a = (long long)(ph + sps * k) * es, b2 = (long long)(ph + sps * k + sps) * es;
        const uint32_t sd = (uint32_t)((int)pi[a] * (int)pq[b2]) - (uint32_t)((int)pi[b2] * (int)pq[a]);
        bit = (int32_t)sd > 0;
      }
      const uint32_t W = __ballot_sync(0xFFFFFFFFu, bit);
      if (lane == 0) B[j] = W;
    }
    if (lane == 0) { B[nw] = 0u; B[nw + 1] = 0u; }
    __syncwarp();
    // search_unique_bit_sequence: first index whose 32 bits equal the access address (btlelib.py:402-412)
    int start = -1;
    for (int j = 0; j < nw && start < 0; ++j) {
      const int s = 32 * j + lane;
      const bool ok = (s + 32 <= num_bit) && (sbits(s) == aa);
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
      if (m) start = 32 * j + __ffs((int)m) - 1;
    }
    if (start >= 0) {
      r_found = 1 + ph;                                    // 1 + the last phase the access address was found on
      r_start = start;
      const int len_info = 8 + num_bit - start;            // 8 zero bits are prepended (btlelib.py:474)
      const uint32_t hdr = sbits(start + 32) ^ wbits(0);   // info[40:] is dewhitened (btlelib.py:265-268)
      const int plen = (int)((hdr >> 8) & (adv ? 0x3Fu : 0x1Fu));        // btlelib.py:477-483
      int crc_start = 40 + 16 + 8 * plen;
      if (crc_start + 24 > len_info) crc_start = len_info - 24;          // btlelib.py:488-490
      const int npdu = crc_start > 40 ? crc_start - 40 : 0;
      r_plen = plen;
      r_npdu = npdu;
      __syncwarp();
      if (lane < 20) {                                     // pdu_bit = info[40:crc_start]
        uint32_t w = 0u;
        const int rem = npdu - 32 * lane;
        if (rem > 0) {
          w = sbits(start + 32 + 32 * lane) ^ wbits(32 * lane);
          if (rem < 32) w &= (1u << rem) - 1u;
        }
        P[lane] = w;
      }
      __syncwarp();
      int ok = 0;
      if (lane == 0) {
        // crc24_core over pdu_bit (btlelib.py:191-219) == reflected CRC-24 on the LSB-first bit stream
        uint32_t crc = crc_init;
        const int nbytes = npdu >> 3;
        for (int b = 0; b < nbytes; ++b) crc = crc_tab[(crc ^ (P[b >> 2] >> (8 * (b & 3)))) & 0xFFu] ^ (crc >> 8);
        for (int b = 8 * nbytes; b < npdu; ++b) {
          const uint32_t fb = (crc ^ (P[b >> 5] >> (b & 31))) & 1u;
          crc = (crc >> 1) ^ (fb ? 0xDA6000u : 0u);
        }
        uint32_t rx = 0;
        if (crc_start >= 40) {
          rx = (sbits(start + crc_start - 8) ^ wbits(crc_start - 40)) & 0xFFFFFFu;
        } else {                                           // CRC window reaches back into the AA / zero bits
          for (int t = 0; t < 24; ++t) {
            const int idx = crc_start + t;
            uint32_t bit = 0;
            if (idx >= 8) bit = (B[(start + idx - 8) >> 5] >> ((start + idx - 8) & 31)) & 1u;
            if (idx >= 40) bit ^= (wh[(idx - 40) >> 5] >> ((idx - 40) & 31)) & 1u;
            rx |= bit << t;
          }
        }
        ok = (crc == rx);
      }
      ok = __shfl_sync(0xFFFFFFFFu, ok, 0);
      r_ok = ok;
      if (ok) { r_phase = ph; break; }                     // btlelib.py:517
    }
    __syncwarp();
  }
  btle_model_rx_rec *o = out + pkt;
  if (lane == 0) {
    o->start = r_start; o->n_pdu_bits = (uint16_t)r_npdu; o->crc_ok = (uint8_t)r_ok; o->phase = (uint8_t)r_phase;
    o->payload_len = (uint8_t)r_plen; o->found = (uint8_t)r_found;
  }
  __syncwarp();
  for (int b = lane; b < 70; b += 32) o->pdu[b] = (uint8_t)(P[b >> 2] >> (8 * (b & 3)));
}

}  // namespace

// ================================================================================================
// C-ABI
// ================================================================================================
struct CfgSlot {                     // one uploaded btle_stream_cfg array + the per-stream parameters derived from it
  btle_stream_cfg *d = nullptr; size_t cap = 0;   // (small LRU cache, see upload_cfgs)
  StreamParams *d_params = nullptr;
  std::vector<StreamParams> host_params;
  std::vector<btle_stream_cfg> host;
  cudaEvent_t last_use = nullptr;
  unsigned long long stamp = 0;
};
struct MapSlot {                     // encoded TMA tensor maps of one (pointer, shape) combination
  const void *ptr = nullptr; size_t n_streams = 0, stride = 0, n_int8 = 0;
  CUtensorMap map32, map12;
  unsigned long long stamp = 0;
};
struct btle_b200_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;    // second stream of the segmented host-buffer path
  std::string err;
  int last_launches = 0;
  bool attr_done = false, attr_sps8_done = false;
  int num_sms = 148;
  void *encode_tiled = nullptr;     // cuTensorMapEncodeTiled, fetched through the runtime
  unsigned long long tick = 0;
  CfgSlot cfg_slot[4];
  MapSlot map_slot[4];
  // scratch owned by the context (host-buffer entry points)
  int8_t *d_iq = nullptr; size_t d_iq_bytes = 0;
  btle_pkt_rec *d_out = nullptr; size_t d_out_cap = 0;
  btle_unit_dir *d_dir = nullptr; size_t d_dir_cap = 0;
  unsigned *d_count = nullptr;
  unsigned *d_count_ring = nullptr; // kCountRing allocation counters for launches that do not hand in their own (no memset node)
  unsigned ring_pos = 0;
  size_t lead_bytes = 0;            // bytes readable in front of d_iq (set by the stream session around its launches; RSSI of hits at a segment's very start)
  unsigned *h_count = nullptr;      // pinned
  btle_pkt_rec *h_recs = nullptr; size_t h_recs_cap = 0;   // pinned staging for records
  btle_unit_dir *h_dir = nullptr; size_t h_dir_cap = 0;    // pinned staging for the unit directory
  int8_t *h_stage[2] = {nullptr, nullptr}; size_t h_stage_bytes = 0;   // pinned staging for pageable callers
  cudaEvent_t stage_free[2] = {nullptr, nullptr};
  void *d_leaf = nullptr; size_t d_leaf_bytes = 0;
  int8_t *d_wide = nullptr; size_t d_wide_bytes = 0;   // wideband capture of the host-buffer channelizer entry points
  btle_wb::Scratch wb;
};

namespace {

#define BTLE_CUDA(ctx, call)                                                              \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                    \
      return BTLE_ECUDA;                                                                  \
    }                                                                                     \
  } while (0)

int ensure(btle_b200_ctx *ctx, void **p, size_t *have, size_t need) {
  if (*have >= need && *p) return BTLE_OK;
  if (*p) cudaFree(*p);
  *p = nullptr; *have = 0;
  const size_t want = need + need / 8 + 4096;
  if (cudaMalloc(p, want) != cudaSuccess) {
    cudaGetLastError();
    ctx->err = "cudaMalloc failed";
    return BTLE_ENOMEM;
  }
  *have = want;
  return BTLE_OK;
}

int validate_cfgs(btle_b200_ctx *ctx, const btle_stream_cfg *cfgs, size_t n) {
  for (size_t i = 0; i < n; ++i)
    if (cfgs[i].channel < 0 || cfgs[i].channel > 39) {   // same range check as btle_rx.c:1432-1435
      ctx->err = "channel number must be within 0~39";
      return BTLE_EINVAL;
    }
  return BTLE_OK;
}

// The cfg array of a launch must live on the device while the kernel runs.  Uploaded arrays are kept in a small
// LRU cache keyed by content; re-using a slot whose last launch may still be running on ANOTHER stream is made safe
// by a stream-side wait on that launch's event (no host or device-wide synchronisation).
constexpr unsigned kCountRing = 64;

int upload_cfgs(btle_b200_ctx *ctx, const btle_stream_cfg *cfgs, size_t n, cudaStream_t st, CfgSlot **slot_out) {
  CfgSlot *pick = nullptr;
  for (CfgSlot &c : ctx->cfg_slot)
    if (c.d && c.host.size() == n && !memcmp(c.host.data(), cfgs, n * sizeof(btle_stream_cfg))) { pick = &c; break; }
  if (!pick) {
    pick = &ctx->cfg_slot[0];
    for (CfgSlot &c : ctx->cfg_slot) if (c.stamp < pick->stamp) pick = &c;
    if (!pick->last_use) BTLE_CUDA(ctx, cudaEventCreateWithFlags(&pick->last_use, cudaEventDisableTiming));
    if (pick->cap < n) {
      if (pick->d) cudaFree(pick->d);                        // (cudaFree waits for work that still uses it)
      if (pick->d_params) cudaFree(pick->d_params);
      pick->d = nullptr; pick->d_params = nullptr; pick->cap = 0;
      const size_t want = n + n / 4 + 16;
      if (cudaMalloc(&pick->d, want * sizeof(btle_stream_cfg)) != cudaSuccess || cudaMalloc(&pick->d_params, want * sizeof(StreamParams)) != cudaSuccess) {
        cudaGetLastError(); ctx->err = "cudaMalloc failed"; return BTLE_ENOMEM;
      }
      pick->cap = want;
    } else if (pick->stamp) {
      BTLE_CUDA(ctx, cudaStreamWaitEvent(st, pick->last_use, 0));
    }
    pick->host.assign(cfgs, cfgs + n);
    pick->host_params.resize(n);
    for (size_t i = 0; i < n; ++i) {                         // make_params(): btle_params.h, the same code the CPU emulator runs
      uint8_t row[48];
      make_whiten_row(cfgs[i].channel, row);
      uint32_t ww[12];
      memcpy(ww, row, 48);
      make_params(cfgs[i], ww, pick->host_params[i]);
    }
    BTLE_CUDA(ctx, cudaMemcpyAsync(pick->d, pick->host.data(), n * sizeof(btle_stream_cfg), cudaMemcpyHostToDevice, st));
    BTLE_CUDA(ctx, cudaMemcpyAsync(pick->d_params, pick->host_params.data(), n * sizeof(StreamParams), cudaMemcpyHostToDevice, st));
  }
  pick->stamp = ++ctx->tick;
  *slot_out = pick;
  return BTLE_OK;
}

// IQ as a 4-D byte tensor {128 B, 2 halves, 256-byte runs, streams}; a box is one half of `rows` consecutive
// runs, so each lane's 256-byte run lands as two conflict-free 128-byte rows.  Encoded maps are cached per
// (pointer, shape): a streaming caller alternates between a few buffers.
int get_maps(btle_b200_ctx *ctx, const int8_t *d_iq, size_t n_streams, size_t stride, size_t n_int8, const MapSlot **out) {
  MapSlot *pick = nullptr;
  for (MapSlot &m : ctx->map_slot)
    if (m.stamp && m.ptr == d_iq && m.n_streams == n_streams && m.stride == stride && m.n_int8 == n_int8) { pick = &m; break; }
  if (!pick) {
    pick = &ctx->map_slot[0];
    for (MapSlot &m : ctx->map_slot) if (m.stamp < pick->stamp) pick = &m;
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    encode_fn enc = reinterpret_cast<encode_fn>(ctx->encode_tiled);
    const cuuint64_t runs = (cuuint64_t)(n_int8 / 256);
    const cuuint64_t dims[4] = {128, 2, runs, (cuuint64_t)n_streams};
    const cuuint64_t strides[3] = {128, 256, (cuuint64_t)(n_streams > 1 ? stride : ((n_int8 + 255) & ~size_t(255)))};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    for (int which = 0; which < 2; ++which) {
      const cuuint32_t box[4] = {128, 1, (cuuint32_t)(which ? kHaloRows : 32), 1};
      const CUresult r = enc(which ? &pick->map12 : &pick->map32, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<int8_t *>(d_iq), dims,
                             strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { pick->stamp = 0; ctx->err = "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"; return BTLE_ECUDA; }
    }
    pick->ptr = d_iq; pick->n_streams = n_streams; pick->stride = stride; pick->n_int8 = n_int8;
  }
  pick->stamp = ++ctx->tick;
  *out = pick;
  return BTLE_OK;
}

Plan plan_for(const btle_b200_ctx *ctx, size_t n_streams, size_t n_int8) {
  return make_plan((long long)n_streams, (long long)(n_int8 / kChunkInt8), ctx->num_sms * kCtasPerSm);
}

// enqueue the persistent kernel for device-resident inputs
int launch_rx(btle_b200_ctx *ctx, const int8_t *d_iq, size_t n_streams, size_t stride, size_t n_int8,
              const btle_stream_cfg *cfgs, btle_pkt_rec *d_out, size_t cap, unsigned *d_count, btle_unit_dir *d_dir,
              cudaStream_t st) {
  ctx->last_launches = 0;
  unsigned *zero_next = nullptr;
  if (d_count) BTLE_CUDA(ctx, cudaMemsetAsync(d_count, 0, sizeof(unsigned), st));
  const long long nchunks = (long long)(n_int8 / kChunkInt8);
  if (nchunks == 0 || n_streams == 0) return BTLE_OK;
  if (!d_count) {
    // no counter from the caller (it reads the unit directory): take the next one of the context's ring.  It is zero —
    // cleared at creation or by the launch kCountRing/2 launches ago — and this launch clears the one used kCountRing/2
    // launches from now (no memset node in front of the kernel; far more launches than that cannot be in flight: every
    // one occupies all SMs).
    d_count = ctx->d_count_ring + ctx->ring_pos;
    zero_next = ctx->d_count_ring + (ctx->ring_pos + kCountRing / 2) % kCountRing;
    ctx->ring_pos = (ctx->ring_pos + 1) % kCountRing;
  }
  const long long spans = (nchunks + kSpanChunks - 1) / kSpanChunks;
  if (spans * (long long)n_streams > 0x07FFFFFFll || nchunks > 0x7FFFFFFFll) { ctx->err = "batch too large for one launch"; return BTLE_EINVAL; }
  const Plan plan = plan_for(ctx, n_streams, n_int8);
  const size_t smem = sizeof(Smem);
  if (!ctx->attr_done) {
    BTLE_CUDA(ctx, cudaFuncSetAttribute(btle_rx_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ctx->attr_done = true;
  }
  CfgSlot *cs = nullptr;
  int rc = upload_cfgs(ctx, cfgs, n_streams, st, &cs);
  if (rc) return rc;
  const MapSlot *ms = nullptr;
  rc = get_maps(ctx, d_iq, n_streams, stride, n_int8, &ms);
  if (rc) return rc;
  const unsigned grid = (unsigned)std::min<long long>(plan.total_units, (long long)ctx->num_sms * kCtasPerSm);   // one persistent CTA per SM
  btle_rx_persistent_kernel<<<grid, kThreads, smem, st>>>(
      ms->map32, ms->map12, d_iq, (long long)stride, (long long)n_int8, cs->d_params, plan, d_out,
      (unsigned)std::min<size_t>(cap, 0xFFFFFFFFu), d_count, reinterpret_cast<uint2 *>(d_dir), zero_next, (long long)ctx->lead_bytes);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaEventRecord(cs->last_use, st));
  ctx->last_launches = 1;
  return BTLE_OK;
}

bool rec_less(const btle_pkt_rec &a, const btle_pkt_rec &b) {
  if (a.stream != b.stream) return a.stream < b.stream;
  if (a.chunk != b.chunk) return a.chunk < b.chunk;
  return a.n0 < b.n0;
}

int ensure_pinned(btle_b200_ctx *ctx, void **p, size_t *have, size_t need) {
  if (*have >= need && *p) return BTLE_OK;
  if (*p) cudaFreeHost(*p);
  *p = nullptr; *have = 0;
  const size_t want = need + need / 4 + 4096;
  if (cudaHostAlloc(p, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); ctx->err = "cudaHostAlloc failed"; return BTLE_ENOMEM; }
  *have = want;
  return BTLE_OK;
}

// memcpy with a few threads: one core moves ~10 GB/s, a PCIe 5 x16 link takes ~55 GB/s
void par_memcpy(void *dst, const void *src, size_t n) {
  const size_t kMin = size_t(4) << 20;
  unsigned t = std::thread::hardware_concurrency();
  t = t >= 16 ? 6 : (t >= 4 ? 2 : 1);
  if (n < 2 * kMin || t < 2) { memcpy(dst, src, n); return; }
  std::vector<std::thread> th;
  const size_t per = ((n / t) + 4095) & ~size_t(4095);
  for (unsigned i = 1; i < t; ++i) {
    const size_t o = std::min(n, i * per), e = std::min(n, (i + 1) * per);
    if (e > o) th.emplace_back([=] { memcpy(static_cast<char *>(dst) + o, static_cast<const char *>(src) + o, e - o); });
  }
  memcpy(dst, src, std::min(n, per));
  for (auto &x : th) x.join();
}

bool is_pinned(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// Host -> device copy of `rows` rows of `width` bytes.  Page-locked sources go straight to the DMA engine; pageable
// sources are moved through two page-locked staging buffers in segments, the CPU copy of segment i+1 overlapping
// the DMA of segment i (cudaMemcpyAsync on pageable memory would stage synchronously at a fraction of the link rate).
int h2d_rows(btle_b200_ctx *ctx, int8_t *dst, size_t dpitch, const int8_t *src, size_t spitch, size_t width, size_t rows,
             cudaStream_t st) {
  if (!width || !rows) return BTLE_OK;
  if (is_pinned(src)) {
    if (rows == 1 || (dpitch == spitch && dpitch == width)) BTLE_CUDA(ctx, cudaMemcpyAsync(dst, src, width * rows, cudaMemcpyHostToDevice, st));
    else BTLE_CUDA(ctx, cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, cudaMemcpyHostToDevice, st));
    return BTLE_OK;
  }
  const size_t seg = size_t(32) << 20;
  if (ctx->h_stage_bytes < seg) {
    for (int b = 0; b < 2; ++b) {
      if (ctx->h_stage[b]) cudaFreeHost(ctx->h_stage[b]);
      ctx->h_stage[b] = nullptr;
      if (cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_stage[b]), seg, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); ctx->err = "cudaHostAlloc failed"; return BTLE_ENOMEM; }
      if (!ctx->stage_free[b]) BTLE_CUDA(ctx, cudaEventCreateWithFlags(&ctx->stage_free[b], cudaEventDisableTiming));
    }
    ctx->h_stage_bytes = seg;
  }
  int b = 0;
  bool used[2] = {false, false};
  for (size_t r = 0; r < rows; ++r)
    for (size_t o = 0; o < width; o += seg) {
      const size_t n = std::min(seg, width - o);
      if (used[b]) BTLE_CUDA(ctx, cudaEventSynchronize(ctx->stage_free[b]));
      par_memcpy(ctx->h_stage[b], src + r * spitch + o, n);
      BTLE_CUDA(ctx, cudaMemcpyAsync(dst + r * dpitch + o, ctx->h_stage[b], n, cudaMemcpyHostToDevice, st));
      BTLE_CUDA(ctx, cudaEventRecord(ctx->stage_free[b], st));
      used[b] = true;
      b ^= 1;
    }
  return BTLE_OK;
}

// After a launch on `st`: count, records and unit directory to the host; records copied into `out` in reference
// order (walk of the directory).  *n_out = packets found (may exceed cap -> BTLE_EOVERFLOW).
int fetch_ordered(btle_b200_ctx *ctx, const btle_pkt_rec *d_out, const btle_unit_dir *d_dir, size_t n_units, btle_pkt_rec *out,
                  size_t cap, size_t *n_out, cudaStream_t st) {
  BTLE_CUDA(ctx, cudaMemcpyAsync(ctx->h_count, ctx->d_count, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  BTLE_CUDA(ctx, cudaStreamSynchronize(st));
  const size_t found = *ctx->h_count;
  const size_t n = std::min(found, cap);
  *n_out = found;
  if (n) {
    size_t hb = ctx->h_recs_cap * sizeof(btle_pkt_rec), db = ctx->h_dir_cap * sizeof(btle_unit_dir);
    int rc = ensure_pinned(ctx, reinterpret_cast<void **>(&ctx->h_recs), &hb, n * sizeof(btle_pkt_rec));
    ctx->h_recs_cap = hb / sizeof(btle_pkt_rec);
    if (rc) return rc;
    rc = ensure_pinned(ctx, reinterpret_cast<void **>(&ctx->h_dir), &db, n_units * sizeof(btle_unit_dir));
    ctx->h_dir_cap = db / sizeof(btle_unit_dir);
    if (rc) return rc;
    BTLE_CUDA(ctx, cudaMemcpyAsync(ctx->h_recs, d_out, n * sizeof(btle_pkt_rec), cudaMemcpyDeviceToHost, st));
    BTLE_CUDA(ctx, cudaMemcpyAsync(ctx->h_dir, d_dir, n_units * sizeof(btle_unit_dir), cudaMemcpyDeviceToHost, st));
    BTLE_CUDA(ctx, cudaStreamSynchronize(st));
    size_t got = 0;
    btle_b200_gather_ordered(ctx->h_recs, n, ctx->h_dir, n_units, out, cap, &got);
  }
  if (found > cap) { ctx->err = "output capacity too small"; return BTLE_EOVERFLOW; }
  return BTLE_OK;
}

int launch_sps8_hits(btle_b200_ctx *ctx, const int16_t *d_iq16, size_t n_samples, uint32_t aa, long long *d_hits, size_t cap, unsigned *d_count,
                     cudaStream_t st) {
  if (!ctx->attr_sps8_done) {
    BTLE_CUDA(ctx, cudaFuncSetAttribute(sps8_hits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSps8Smem));
    ctx->attr_sps8_done = true;
  }
  const long long groups = ((long long)n_samples + 255) / 256, tiles = (groups + kSps8Groups - 1) / kSps8Groups;
  const unsigned grid = kSps8Bufs > 1 ? (unsigned)std::min<long long>(tiles, 3ll * ctx->num_sms) : (unsigned)std::min<long long>(tiles, 0x7FFFFFFF);
  sps8_hits_kernel<<<grid, 256, kSps8Smem, st>>>(d_iq16, (long long)n_samples, tiles, aa, d_hits, (unsigned)cap, d_count);
  BTLE_CUDA(ctx, cudaGetLastError());
  return BTLE_OK;
}

int leaf_buf(btle_b200_ctx *ctx, size_t bytes) { return ensure(ctx, &ctx->d_leaf, &ctx->d_leaf_bytes, bytes); }

}  // namespace

extern "C" {

uint32_t btle_b200_version(void) { return (0u << 16) | 1u; }

const char *btle_b200_strerror(int code) {
  switch (code) {
    case BTLE_OK: return "ok";
    case BTLE_EINVAL: return "invalid argument";
    case BTLE_ENODEV: return "no usable CUDA device";
    case BTLE_ENOMEM: return "out of memory";
    case BTLE_ECUDA: return "CUDA error";
    case BTLE_EOVERFLOW: return "more packets than the output capacity";
    default: return "unknown error";
  }
}

const char *btle_b200_last_error(const btle_b200_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
int btle_b200_last_launches(const btle_b200_ctx *ctx) { return ctx ? ctx->last_launches : 0; }

int btle_b200_bind_host_numa(int cuda_device, int *node_out) {
  if (node_out) *node_out = -1;
  char bus[64] = {0};
  if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, cuda_device) != cudaSuccess) { cudaGetLastError(); return BTLE_ENODEV; }
  for (char *c = bus; *c; ++c) if (*c >= 'A' && *c <= 'F') *c = (char)(*c - 'A' + 'a');
  char path[256];
  snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
  int node = -1;
  if (FILE *f = fopen(path, "r")) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
  if (node < 0) return BTLE_OK;                            // single-node machine or not exposed: nothing to bind
  snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
  cpu_set_t want, have, both;
  CPU_ZERO(&want);
  if (FILE *f = fopen(path, "r")) {                        // "0-47,96-143"
    int a, b;
    while (fscanf(f, "%d", &a) == 1) {
      b = a;
      int ch = fgetc(f);
      if (ch == '-') { if (fscanf(f, "%d", &b) != 1) b = a; ch = fgetc(f); }
      for (int c = a; c <= b && c < CPU_SETSIZE; ++c) CPU_SET(c, &want);
      if (ch != ',') break;
    }
    fclose(f);
  }
  if (sched_getaffinity(0, sizeof have, &have) == 0) {
    CPU_AND(&both, &want, &have);                          // never widen what a cpuset / taskset allowed
    if (CPU_COUNT(&both) > 0) sched_setaffinity(0, sizeof both, &both);
  }
  if (node < 1024) {                                       // MPOL_PREFERRED: pages this thread touches (and pins) come from `node`
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(8 * sizeof mask));
  }
  if (node_out) *node_out = node;
  return BTLE_OK;
}

int btle_b200_create(btle_b200_ctx **out, int cuda_device) {
  if (!out) return BTLE_EINVAL;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || cuda_device < 0 || cuda_device >= ndev) {
    cudaGetLastError();
    return BTLE_ENODEV;   // no CPU fallback, by design
  }
  btle_b200_ctx *ctx = new (std::nothrow) btle_b200_ctx();
  if (!ctx) return BTLE_ENOMEM;
  ctx->device = cuda_device;
  if (cudaSetDevice(cuda_device) != cudaSuccess) { delete ctx; return BTLE_ENODEV; }
  // protocol tables -> constant memory
  uint32_t ww[40][12];
  for (int ch = 0; ch < 40; ++ch) { uint8_t row[48]; make_whiten_row(ch, row); memcpy(ww[ch], row, 48); }
  uint32_t crc[1024];
  make_crc4(crc);
  if (cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, cuda_device) != cudaSuccess || ctx->num_sms < 1) {
    cudaGetLastError();
    delete ctx;
    return BTLE_ECUDA;
  }
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ctx->encode_tiled, cudaEnableDefault, nullptr) != cudaSuccess ||
      !ctx->encode_tiled) {
    cudaGetLastError();
    delete ctx;
    return BTLE_ENODEV;
  }
  {
    static int8_t c1[1024], s1[1024], c2[2048], s2[2048];
    const double two_pi = 6.283185307179586476925286766559;
    for (int k = 0; k < 1024; ++k) { c1[k] = (int8_t)nearbyint(127.0 * cos(two_pi * k / 1024.0)); s1[k] = (int8_t)nearbyint(127.0 * sin(two_pi * k / 1024.0)); }
    for (int k = 0; k < 2048; ++k) { c2[k] = (int8_t)nearbyint(127.0 * cos(two_pi * k / 2048.0)); s2[k] = (int8_t)nearbyint(127.0 * sin(two_pi * k / 2048.0)); }
    if (cudaMemcpyToSymbol(c_cos1024, c1, sizeof c1) != cudaSuccess || cudaMemcpyToSymbol(c_sin1024, s1, sizeof s1) != cudaSuccess ||
        cudaMemcpyToSymbol(c_cos2048, c2, sizeof c2) != cudaSuccess || cudaMemcpyToSymbol(c_sin2048, s2, sizeof s2) != cudaSuccess) {
      cudaGetLastError();
      btle_b200_destroy(ctx);
      return BTLE_ECUDA;
    }
  }
  uint32_t thr[13];
  for (int k = 0; k < 13; ++k) {                         // P(round(N(-0.3, 0.8)) <= v), v = -7 + k
    const double p = 0.5 * erfc(-(((double)(-7 + k) + 0.5 + 0.3) / 0.8) / sqrt(2.0));
    thr[k] = (uint32_t)std::min(4294967295.0, p * 4294967296.0);
  }
  if (cudaMemcpyToSymbol(c_noise_thr, thr, sizeof thr) != cudaSuccess ||
      cudaMemcpyToSymbol(c_whiten_words, ww, sizeof ww) != cudaSuccess ||
      cudaMemcpyToSymbol(c_crc4, crc, sizeof crc) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMalloc(&ctx->d_count, sizeof(unsigned)) != cudaSuccess ||
      cudaMalloc(&ctx->d_count_ring, 64 * sizeof(unsigned)) != cudaSuccess || cudaMemset(ctx->d_count_ring, 0, 64 * sizeof(unsigned)) != cudaSuccess ||
      cudaHostAlloc(&ctx->h_count, sizeof(unsigned), cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    btle_b200_destroy(ctx);
    return BTLE_ECUDA;
  }
  *out = ctx;
  return BTLE_OK;
}

void btle_b200_destroy(btle_b200_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  cudaFree(ctx->d_iq); cudaFree(ctx->d_out); cudaFree(ctx->d_dir); cudaFree(ctx->d_count); cudaFree(ctx->d_count_ring); cudaFree(ctx->d_leaf);
  cudaFree(ctx->d_wide);
  btle_wb::release(&ctx->wb);
  for (CfgSlot &c : ctx->cfg_slot) { cudaFree(c.d); cudaFree(c.d_params); if (c.last_use) cudaEventDestroy(c.last_use); }
  if (ctx->h_count) cudaFreeHost(ctx->h_count);
  if (ctx->h_recs) cudaFreeHost(ctx->h_recs);
  if (ctx->h_dir) cudaFreeHost(ctx->h_dir);
  for (int b = 0; b < 2; ++b) { if (ctx->h_stage[b]) cudaFreeHost(ctx->h_stage[b]); if (ctx->stage_free[b]) cudaEventDestroy(ctx->stage_free[b]); }
  delete ctx;
}

size_t btle_b200_rx_units(const btle_b200_ctx *ctx, size_t n_streams, size_t n_int8) {
  if (!ctx || !n_streams || n_int8 < (size_t)kChunkInt8) return 0;
  return (size_t)plan_for(ctx, n_streams, n_int8).total_units;
}

int btle_b200_rx_device_dir(btle_b200_ctx *ctx, const int8_t *d_iq, size_t n_streams, size_t stride, size_t n_int8,
                            const btle_stream_cfg *cfgs, btle_pkt_rec *d_out, size_t cap, uint32_t *d_count,
                            btle_unit_dir *d_dir, size_t dir_cap, void *cuda_stream) {
  if (!ctx || (!d_out && cap) || (!cfgs && n_streams) || !d_dir) return BTLE_EINVAL;
  if ((reinterpret_cast<uintptr_t>(d_iq) & 15) || (n_streams > 1 && (stride & 15))) { ctx->err = "device IQ must be 16-byte aligned"; return BTLE_EINVAL; }
  if (dir_cap < btle_b200_rx_units(ctx, n_streams, n_int8)) { ctx->err = "unit directory too small (btle_b200_rx_units)"; return BTLE_EINVAL; }
  int rc = validate_cfgs(ctx, cfgs, n_streams);
  if (rc) return rc;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  return launch_rx(ctx, d_iq, n_streams, stride, n_int8, cfgs, d_out, cap, d_count, d_dir, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int btle_b200_rx_device(btle_b200_ctx *ctx, const int8_t *d_iq, size_t n_streams, size_t stride, size_t n_int8,
                        const btle_stream_cfg *cfgs, btle_pkt_rec *d_out, size_t cap, uint32_t *d_count,
                        void *cuda_stream) {
  if (!ctx) return BTLE_EINVAL;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  // the directory goes to context-owned scratch (callers of this entry point sort the records themselves)
  const size_t units = btle_b200_rx_units(ctx, n_streams, n_int8);
  size_t have = ctx->d_dir_cap * sizeof(btle_unit_dir);
  const int rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_dir), &have, std::max<size_t>(units, 1) * sizeof(btle_unit_dir));
  ctx->d_dir_cap = have / sizeof(btle_unit_dir);
  if (rc) return rc;
  return btle_b200_rx_device_dir(ctx, d_iq, n_streams, stride, n_int8, cfgs, d_out, cap, d_count, ctx->d_dir, ctx->d_dir_cap, cuda_stream);
}

void btle_b200_sort_records(btle_pkt_rec *recs, size_t n) { std::sort(recs, recs + n, rec_less); }

int btle_b200_gather_ordered(const btle_pkt_rec *recs, size_t n_recs, const btle_unit_dir *dir, size_t n_units,
                             btle_pkt_rec *out, size_t cap, size_t *n_out) {
  if ((!recs && n_recs) || (!dir && n_units) || (!out && cap) || !n_out) return BTLE_EINVAL;
  size_t pos = 0, total = 0;
  for (size_t u = 0; u < n_units; ++u) {
    const size_t base = dir[u].base, cnt = dir[u].count;
    total += cnt;
    if (base >= n_recs) continue;                           // block was cut off by the producer's capacity
    const size_t take = std::min(std::min(cnt, n_recs - base), cap - pos);
    if (take) memcpy(out + pos, recs + base, take * sizeof(btle_pkt_rec));
    pos += take;
  }
  *n_out = total;
  return total > cap || pos < total ? BTLE_EOVERFLOW : BTLE_OK;
}

int btle_b200_rx_batch(btle_b200_ctx *ctx, const int8_t *iq, size_t n_streams, size_t stride, size_t n_int8,
                       const btle_stream_cfg *cfgs, btle_pkt_rec *out, size_t cap, size_t *n_out) {
  if (!ctx || !n_out || (!out && cap) || (!cfgs && n_streams) || (!iq && n_streams && n_int8)) return BTLE_EINVAL;
  *n_out = 0;
  if (n_streams > 1 && stride < n_int8) { ctx->err = "stream stride smaller than stream length"; return BTLE_EINVAL; }
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t pitch = (n_int8 + 15) & ~size_t(15);
  int rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_iq), &ctx->d_iq_bytes, std::max<size_t>(pitch * n_streams, 16));
  if (rc) return rc;
  size_t out_bytes = ctx->d_out_cap * sizeof(btle_pkt_rec);
  rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_out), &out_bytes, std::max<size_t>(cap, 1) * sizeof(btle_pkt_rec));
  ctx->d_out_cap = out_bytes / sizeof(btle_pkt_rec);
  if (rc) return rc;
  // exactly the caller's bytes are read: n_int8 per capture, never the padding behind the last one
  rc = h2d_rows(ctx, ctx->d_iq, pitch, iq, n_streams > 1 ? stride : n_int8, n_int8, n_streams, st);
  if (rc) return rc;
  rc = btle_b200_rx_device(ctx, ctx->d_iq, n_streams, pitch, n_int8, cfgs, ctx->d_out, cap, ctx->d_count, st);
  if (rc) return rc;
  return fetch_ordered(ctx, ctx->d_out, ctx->d_dir, btle_b200_rx_units(ctx, n_streams, n_int8), out, cap, n_out, st);
}

int btle_b200_rx_iq16(btle_b200_ctx *ctx, const int16_t *iq16, size_t n_int16, int shift, const btle_stream_cfg *cfg,
                      btle_pkt_rec *out, size_t cap, size_t *n_out) {
  if (!ctx || (!iq16 && n_int16) || !cfg || !n_out || (!out && cap) || shift < 0 || shift > 8) return BTLE_EINVAL;
  *n_out = 0;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t pitch = (n_int16 + 255) & ~size_t(255);
  int rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_iq), &ctx->d_iq_bytes, pitch + 2 * n_int16 + 512);
  if (rc) return rc;
  int16_t *d16 = reinterpret_cast<int16_t *>(ctx->d_iq + pitch + 256);      // behind the int8 capture
  size_t out_bytes = ctx->d_out_cap * sizeof(btle_pkt_rec);
  rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_out), &out_bytes, std::max<size_t>(cap, 1) * sizeof(btle_pkt_rec));
  ctx->d_out_cap = out_bytes / sizeof(btle_pkt_rec);
  if (rc) return rc;
  if (n_int16) {
    rc = h2d_rows(ctx, reinterpret_cast<int8_t *>(d16), 2 * n_int16, reinterpret_cast<const int8_t *>(iq16), 2 * n_int16, 2 * n_int16, 1, st);
    if (rc) return rc;
    iq16_to_iq8_kernel<<<(unsigned)std::min<size_t>((n_int16 + 255) / 256, 148 * 16), 256, 0, st>>>(d16, (long long)n_int16, shift, ctx->d_iq);
    BTLE_CUDA(ctx, cudaGetLastError());
  }
  rc = btle_b200_rx_device(ctx, ctx->d_iq, 1, pitch, n_int16, cfg, ctx->d_out, cap, ctx->d_count, st);
  if (rc) return rc;
  return fetch_ordered(ctx, ctx->d_out, ctx->d_dir, btle_b200_rx_units(ctx, 1, n_int16), out, cap, n_out, st);
}

// ---- wideband captures: channelizer (btle_wideband.cu) in front of the receiver -------------------------------------
static int wideband_check(btle_b200_ctx *ctx, size_t n_samples, const btle_wideband_cfg *cfg, const int32_t *channels, size_t n_ch,
                          size_t out_stride) {
  if (!cfg) { ctx->err = "wideband cfg is NULL"; return BTLE_EINVAL; }
  const int rc = btle_wb::validate(*cfg, channels, n_ch, &ctx->err);
  if (rc) return rc;
  if (out_stride & 15) { ctx->err = "channel output stride must be a multiple of 16"; return BTLE_EINVAL; }
  if (n_ch && out_stride < 2 * btle_wb::out_samples(n_samples, cfg->decim)) {
    ctx->err = "channel output stride " + std::to_string(out_stride) + " is smaller than 2*ceil(n_samples/decim) = " +
               std::to_string(2 * btle_wb::out_samples(n_samples, cfg->decim));
    return BTLE_EINVAL;
  }
  return BTLE_OK;
}

// host capture -> context scratch (d_wide) -> channels in ctx->d_iq, rows of out_stride bytes; enqueued on `st`
static int wideband_stage(btle_b200_ctx *ctx, const int8_t *wide, size_t n_samples, const btle_wideband_cfg &cfg, const int32_t *channels,
                          size_t n_ch, size_t out_stride, cudaStream_t st) {
  int rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_wide), &ctx->d_wide_bytes, std::max<size_t>(2 * n_samples, 16));
  if (rc) return rc;
  rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_iq), &ctx->d_iq_bytes, std::max<size_t>(n_ch * out_stride, 16));
  if (rc) return rc;
  rc = h2d_rows(ctx, ctx->d_wide, 2 * n_samples, wide, 2 * n_samples, 2 * n_samples, 1, st);
  if (rc) return rc;
  return btle_wb::launch(&ctx->wb, ctx->d_wide, n_samples, cfg, channels, n_ch, ctx->d_iq, out_stride, st, &ctx->err);
}

int btle_b200_wideband_taps(const btle_wideband_cfg *cfg, int channel, int16_t *taps, size_t cap, size_t *n_taps, int *out_shift) {
  if (!cfg || !n_taps || (!taps && cap)) return BTLE_EINVAL;
  std::string err;
  std::vector<int16_t> h;
  int shift = 0;
  const int rc = btle_wb::channel_taps(*cfg, channel, &h, &shift, &err);
  if (rc) return rc;
  *n_taps = h.size() / 2;
  if (out_shift) *out_shift = shift;
  if (cap < *n_taps) return BTLE_EOVERFLOW;
  memcpy(taps, h.data(), h.size() * sizeof(int16_t));
  return BTLE_OK;
}

int btle_b200_channelize_device(btle_b200_ctx *ctx, const int8_t *d_wide, size_t n_samples, const btle_wideband_cfg *cfg,
                                const int32_t *channels, size_t n_ch, int8_t *d_out, size_t out_stride, void *cuda_stream) {
  if (!ctx) return BTLE_EINVAL;
  int rc = wideband_check(ctx, n_samples, cfg, channels, n_ch, out_stride);
  if (rc) return rc;
  if ((!d_wide && n_samples) || (!d_out && n_ch)) { ctx->err = "device buffer is NULL"; return BTLE_EINVAL; }
  if ((reinterpret_cast<uintptr_t>(d_wide) & 15) || (reinterpret_cast<uintptr_t>(d_out) & 15)) {
    ctx->err = "device wideband input and channel output must be 16-byte aligned";
    return BTLE_EINVAL;
  }
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  return btle_wb::launch(&ctx->wb, d_wide, n_samples, *cfg, channels, n_ch, d_out, out_stride, reinterpret_cast<cudaStream_t>(cuda_stream),
                         &ctx->err);
}

int btle_b200_channelize(btle_b200_ctx *ctx, const int8_t *wide, size_t n_samples, const btle_wideband_cfg *cfg, const int32_t *channels,
                         size_t n_ch, int8_t *out, size_t out_stride) {
  if (!ctx) return BTLE_EINVAL;
  int rc = wideband_check(ctx, n_samples, cfg, channels, n_ch, out_stride);
  if (rc) return rc;
  if ((!wide && n_samples) || (!out && n_ch)) { ctx->err = "host buffer is NULL"; return BTLE_EINVAL; }
  if (!n_ch || !n_samples) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  rc = wideband_stage(ctx, wide, n_samples, *cfg, channels, n_ch, out_stride, st);
  if (rc) return rc;
  const size_t width = 2 * btle_wb::out_samples(n_samples, cfg->decim);   // the padding of each row is left as it is
  BTLE_CUDA(ctx, cudaMemcpy2DAsync(out, out_stride, ctx->d_iq, out_stride, width, n_ch, cudaMemcpyDeviceToHost, st));
  BTLE_CUDA(ctx, cudaStreamSynchronize(st));
  return BTLE_OK;
}

int btle_b200_rx_wideband(btle_b200_ctx *ctx, const int8_t *wide, size_t n_samples, const btle_wideband_cfg *cfg,
                          const btle_stream_cfg *cfgs, size_t n_ch, btle_pkt_rec *out, size_t cap, size_t *n_out) {
  if (!ctx || !n_out || (!out && cap) || (!cfgs && n_ch) || (!wide && n_samples)) return BTLE_EINVAL;
  *n_out = 0;
  if (!cfg) { ctx->err = "wideband cfg is NULL"; return BTLE_EINVAL; }
  std::vector<int32_t> channels(n_ch);
  for (size_t i = 0; i < n_ch; ++i) channels[i] = cfgs[i].channel;
  const size_t n_int8 = 2 * btle_wb::out_samples(n_samples, std::max(cfg->decim, 1)), stride = (n_int8 + 15) & ~size_t(15);
  int rc = wideband_check(ctx, n_samples, cfg, channels.data(), n_ch, stride);
  if (rc) return rc;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  size_t out_bytes = ctx->d_out_cap * sizeof(btle_pkt_rec);
  rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_out), &out_bytes, std::max<size_t>(cap, 1) * sizeof(btle_pkt_rec));
  ctx->d_out_cap = out_bytes / sizeof(btle_pkt_rec);
  if (rc) return rc;
  if (n_ch && n_samples) {
    rc = wideband_stage(ctx, wide, n_samples, *cfg, channels.data(), n_ch, stride, st);
    if (rc) return rc;
  }
  rc = btle_b200_rx_device(ctx, ctx->d_iq, n_ch, stride, n_int8, cfgs, ctx->d_out, cap, ctx->d_count, st);
  if (rc) return rc;
  return fetch_ordered(ctx, ctx->d_out, ctx->d_dir, btle_b200_rx_units(ctx, n_ch, n_int8), out, cap, n_out, st);
}

int btle_b200_rx(btle_b200_ctx *ctx, const int8_t *iq, size_t n_int8, const btle_stream_cfg *cfg, btle_pkt_rec *out,
                 size_t cap, size_t *n_out) {
  return btle_b200_rx_batch(ctx, iq, 1, n_int8, n_int8, cfg, out, cap, n_out);
}

// ---- streaming session: one capture of unbounded length, pushed in pieces ---------------------------------------
}  // extern "C"

struct btle_b200_stream {
  btle_b200_ctx *ctx = nullptr;
  btle_stream_cfg cfg{};
  size_t seg_chunks = 0, seg_bytes = 0, buf_bytes = 0;     // a segment = seg_chunks chunks (+ kLook look-ahead bytes behind it)
  static constexpr size_t kLook = 4096;                    // >= 3008 + the kernel's 12-group tile (3072 + 4)
  static constexpr size_t kLead = 256;                     // bytes of the previous segment kept in front (a hit may start up to 124 samples
                                                           // before its chunk; the RSSI sum reads the raw IQ there)
  struct Half {
    int8_t *h = nullptr, *d = nullptr;                     // page-locked host / device IQ buffers
    btle_pkt_rec *d_out = nullptr; btle_unit_dir *d_dir = nullptr; unsigned *d_count = nullptr;
    unsigned *h_count = nullptr; btle_unit_dir *h_dir = nullptr; btle_pkt_rec *h_recs = nullptr;
    size_t cap = 0, units = 0, fill = 0, n_submitted = 0;
    long long first_chunk = 0;
    cudaStream_t st = nullptr;
    bool busy = false;
  } half[2];
  int cur = 0;                                             // half being filled
  long long next_chunk = 0;                                // stream-wide index of the first chunk of the half being filled
  std::vector<btle_pkt_rec> ready;                         // decoded, not yet handed out
  size_t ready_pos = 0;
};

namespace {
int stream_submit(btle_b200_stream *s, int b, size_t n_int8) {
  btle_b200_ctx *ctx = s->ctx;
  auto &H = s->half[b];
  H.n_submitted = n_int8;
  H.first_chunk = s->next_chunk;
  if (n_int8 < (size_t)kChunkInt8) { H.busy = false; return BTLE_OK; }
  constexpr size_t L = btle_b200_stream::kLead;
  BTLE_CUDA(ctx, cudaMemcpyAsync(H.d, H.h, L + n_int8, cudaMemcpyHostToDevice, H.st));
  ctx->lead_bytes = L;
  const int rc = btle_b200_rx_device_dir(ctx, H.d + L, 1, s->buf_bytes, n_int8, &s->cfg, H.d_out, H.cap, H.d_count, H.d_dir, H.units, H.st);
  ctx->lead_bytes = 0;
  if (rc) return rc;
  BTLE_CUDA(ctx, cudaMemcpyAsync(H.h_count, H.d_count, sizeof(unsigned), cudaMemcpyDeviceToHost, H.st));
  BTLE_CUDA(ctx, cudaMemcpyAsync(H.h_dir, H.d_dir, H.units * sizeof(btle_unit_dir), cudaMemcpyDeviceToHost, H.st));
  H.busy = true;
  return BTLE_OK;
}
// wait for a submitted half, append its records (reference order, stream-wide chunk numbers) to s->ready
int stream_collect(btle_b200_stream *s, int b) {
  btle_b200_ctx *ctx = s->ctx;
  auto &H = s->half[b];
  if (!H.busy) return BTLE_OK;
  H.busy = false;
  BTLE_CUDA(ctx, cudaStreamSynchronize(H.st));
  const size_t found = *H.h_count;
  if (found > H.cap) { ctx->err = "stream segment produced more packets than BTLE_MAX_PKTS_PER_CHUNK allows"; return BTLE_EOVERFLOW; }
  if (!found) return BTLE_OK;
  BTLE_CUDA(ctx, cudaMemcpyAsync(H.h_recs, H.d_out, found * sizeof(btle_pkt_rec), cudaMemcpyDeviceToHost, H.st));
  BTLE_CUDA(ctx, cudaStreamSynchronize(H.st));
  const size_t units = btle_b200_rx_units(ctx, 1, H.n_submitted);
  const size_t at = s->ready.size();
  s->ready.resize(at + found);
  size_t got = 0;
  btle_b200_gather_ordered(H.h_recs, found, H.h_dir, units, s->ready.data() + at, found, &got);
  for (size_t i = at; i < at + found; ++i) s->ready[i].chunk += (int32_t)H.first_chunk;
  return BTLE_OK;
}
size_t stream_take(btle_b200_stream *s, btle_pkt_rec *out, size_t cap) {
  const size_t n = std::min(cap, s->ready.size() - s->ready_pos);
  if (n) memcpy(out, s->ready.data() + s->ready_pos, n * sizeof(btle_pkt_rec));
  s->ready_pos += n;
  if (s->ready_pos == s->ready.size()) { s->ready.clear(); s->ready_pos = 0; }
  return n;
}
}  // namespace

extern "C" {

int btle_b200_stream_open(btle_b200_ctx *ctx, const btle_stream_cfg *cfg, size_t segment_chunks, btle_b200_stream **out) {
  if (!ctx || !cfg || !out) return BTLE_EINVAL;
  *out = nullptr;
  int rc = validate_cfgs(ctx, cfg, 1);
  if (rc) return rc;
  if (segment_chunks == 0) segment_chunks = 4096;           // 64 MiB of IQ = 8.4 s of air per segment
  if (segment_chunks > (1u << 20)) { ctx->err = "segment too large"; return BTLE_EINVAL; }
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  btle_b200_stream *s = new (std::nothrow) btle_b200_stream();
  if (!s) return BTLE_ENOMEM;
  s->ctx = ctx; s->cfg = *cfg; s->seg_chunks = segment_chunks; s->seg_bytes = segment_chunks * (size_t)kChunkInt8;
  s->buf_bytes = s->seg_bytes + btle_b200_stream::kLook;
  for (auto &H : s->half) {
    H.cap = segment_chunks * (BTLE_MAX_PKTS_PER_CHUNK + 16);
    H.units = btle_b200_rx_units(ctx, 1, s->buf_bytes) + 1;
    if (cudaHostAlloc(reinterpret_cast<void **>(&H.h), btle_b200_stream::kLead + s->buf_bytes, cudaHostAllocDefault) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void **>(&H.d), btle_b200_stream::kLead + s->buf_bytes) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void **>(&H.d_out), H.cap * sizeof(btle_pkt_rec)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void **>(&H.d_dir), H.units * sizeof(btle_unit_dir)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void **>(&H.d_count), sizeof(unsigned)) != cudaSuccess ||
        cudaHostAlloc(reinterpret_cast<void **>(&H.h_count), sizeof(unsigned), cudaHostAllocDefault) != cudaSuccess ||
        cudaHostAlloc(reinterpret_cast<void **>(&H.h_dir), H.units * sizeof(btle_unit_dir), cudaHostAllocDefault) != cudaSuccess ||
        cudaHostAlloc(reinterpret_cast<void **>(&H.h_recs), H.cap * sizeof(btle_pkt_rec), cudaHostAllocDefault) != cudaSuccess ||
        cudaStreamCreateWithFlags(&H.st, cudaStreamNonBlocking) != cudaSuccess) {
      cudaGetLastError();
      ctx->err = "stream_open: allocation failed";
      btle_b200_stream_close(s);
      return BTLE_ENOMEM;
    }
    memset(H.h, 0, btle_b200_stream::kLead);                // nothing before the start of the stream
  }
  *out = s;
  return BTLE_OK;
}

void btle_b200_stream_close(btle_b200_stream *s) {
  if (!s) return;
  cudaSetDevice(s->ctx->device);
  for (auto &H : s->half) {
    if (H.st) { cudaStreamSynchronize(H.st); cudaStreamDestroy(H.st); }
    if (H.h) cudaFreeHost(H.h);
    if (H.h_count) cudaFreeHost(H.h_count);
    if (H.h_dir) cudaFreeHost(H.h_dir);
    if (H.h_recs) cudaFreeHost(H.h_recs);
    cudaFree(H.d); cudaFree(H.d_out); cudaFree(H.d_dir); cudaFree(H.d_count);
  }
  delete s;
}

int btle_b200_stream_set_cfg(btle_b200_stream *s, const btle_stream_cfg *cfg) {
  if (!s || !cfg) return BTLE_EINVAL;
  const int rc = validate_cfgs(s->ctx, cfg, 1);
  if (rc) return rc;
  s->cfg = *cfg;                                            // used from the next submitted segment on
  return BTLE_OK;
}

int btle_b200_stream_acquire(btle_b200_stream *s, int8_t **buf, size_t *space) {
  if (!s || !buf || !space) return BTLE_EINVAL;
  auto &H = s->half[s->cur];
  *buf = H.h + btle_b200_stream::kLead + H.fill;
  *space = s->buf_bytes - H.fill;
  return BTLE_OK;
}

int btle_b200_stream_commit(btle_b200_stream *s, size_t n_int8, btle_pkt_rec *out, size_t cap, size_t *n_out) {
  if (!s || !n_out || (!out && cap)) return BTLE_EINVAL;
  *n_out = 0;
  auto &H = s->half[s->cur];
  if (n_int8 > s->buf_bytes - H.fill) { s->ctx->err = "stream_commit: more bytes than acquired"; return BTLE_EINVAL; }
  BTLE_CUDA(s->ctx, cudaSetDevice(s->ctx->device));
  H.fill += n_int8;
  if (H.fill == s->buf_bytes) {                             // segment + look-ahead complete: hand it to the GPU
    const int b = s->cur, o = b ^ 1;
    int rc = stream_collect(s, o);                          // the other half's previous segment must be done before its buffers are reused
    if (rc) return rc;
    rc = stream_submit(s, b, s->buf_bytes);
    if (rc) return rc;
    // the look-ahead bytes are the beginning of the next segment, the bytes in front of them its lead
    memcpy(s->half[o].h, H.h + s->seg_bytes, btle_b200_stream::kLead + btle_b200_stream::kLook);
    s->half[o].fill = btle_b200_stream::kLook;
    s->next_chunk += (long long)s->seg_chunks;
    s->cur = o;
  }
  *n_out = stream_take(s, out, cap);
  return BTLE_OK;
}

int btle_b200_stream_push(btle_b200_stream *s, const int8_t *iq, size_t n_int8, btle_pkt_rec *out, size_t cap, size_t *n_out) {
  if (!s || (!iq && n_int8) || !n_out || (!out && cap)) return BTLE_EINVAL;
  *n_out = 0;
  size_t done = 0;
  while (done < n_int8) {
    int8_t *buf; size_t space;
    btle_b200_stream_acquire(s, &buf, &space);
    const size_t n = std::min(space, n_int8 - done);
    memcpy(buf, iq + done, n);
    done += n;
    size_t got = 0;
    const int rc = btle_b200_stream_commit(s, n, out + *n_out, cap - *n_out, &got);
    *n_out += got;
    if (rc) return rc;
  }
  return BTLE_OK;
}

int btle_b200_stream_finish(btle_b200_stream *s, btle_pkt_rec *out, size_t cap, size_t *n_out) {
  if (!s || !n_out || (!out && cap)) return BTLE_EINVAL;
  *n_out = 0;
  BTLE_CUDA(s->ctx, cudaSetDevice(s->ctx->device));
  const int b = s->cur, o = b ^ 1;
  int rc = stream_collect(s, o);
  if (rc) return rc;
  auto &H = s->half[b];
  if (H.fill >= (size_t)kChunkInt8) {                       // the tail: complete chunks only, bytes behind them are look-ahead
    rc = stream_submit(s, b, H.fill);
    if (rc) return rc;
    rc = stream_collect(s, b);
    if (rc) return rc;
    s->next_chunk += (long long)(H.fill / kChunkInt8);
  }
  H.fill = 0;
  *n_out = stream_take(s, out, cap);
  return (s->ready.size() > s->ready_pos) ? BTLE_EOVERFLOW : BTLE_OK;   // call again with more room
}

// ---- leaf functions ------------------------------------------------------------------------------
int btle_b200_dbits(btle_b200_ctx *ctx, const int8_t *iq, size_t n_samples, uint8_t *d_out) {
  if (!ctx || !iq || !d_out) return BTLE_EINVAL;
  if (n_samples == 0) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t in_bytes = 2 * n_samples + 2, in_al = (in_bytes + 255) & ~size_t(255);
  int rc = leaf_buf(ctx, in_al + n_samples);
  if (rc) return rc;
  int8_t *d_in = static_cast<int8_t *>(ctx->d_leaf);
  uint8_t *d_d = reinterpret_cast<uint8_t *>(d_in) + in_al;
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_in, iq, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
  dbits_kernel<<<(unsigned)((n_samples + 255) / 256), 256, 0, ctx->stream>>>(d_in, (long long)n_samples, d_d);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_out, d_d, n_samples, cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

int btle_b200_search_unique_bits(btle_b200_ctx *ctx, const int8_t *rxp, int search_len, const uint8_t *unique_bits,
                                 const uint8_t *unique_bits_mask, int num_bits) {
  // hits are even values >= -248 and -1 means "none" (btle_rx.c:1550/:1561): errors are reported as
  // BTLE_SEARCH_ERR(code) = code - 1000 so that no error can be mistaken for a result
  if (!ctx || !rxp || !unique_bits || !unique_bits_mask || num_bits != 32 || search_len < 0 || search_len > 4096)
    return BTLE_SEARCH_ERR(BTLE_EINVAL);      // the reference only ever passes LEN_DEMOD_BUF_ACCESS = 32
  if (search_len == 0) return -1;
#define BTLE_CUDA_S(ctx, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_); return BTLE_SEARCH_ERR(BTLE_ECUDA); } } while (0)
  BTLE_CUDA_S(ctx, cudaSetDevice(ctx->device));
  btle_stream_cfg cfg{};
  cfg.channel = 37;
  for (int p = 0; p < 32; ++p) {
    cfg.access_addr |= (uint32_t)(unique_bits[p] & 1u) << p;
    cfg.access_mask |= (uint32_t)(unique_bits_mask[p] ? 1u : 0u) << p;
  }
  const size_t valid = 8 * (size_t)search_len + 2;          // int8 the reference reads (:1528-1529)
  const int ngroups = (int)((4 * (size_t)search_len + 127) / 128);
  const size_t in_al = ((size_t)ngroups * 256 + 16 + 255) & ~size_t(255);
  int rc = leaf_buf(ctx, in_al + ((size_t)ngroups + 1) * 20 + 16);
  if (rc) return BTLE_SEARCH_ERR(rc);
  int8_t *d_in = static_cast<int8_t *>(ctx->d_leaf);
  uint32_t *d_pd = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(d_in) + in_al);
  uint32_t *d_cand = d_pd + 4 * ((size_t)ngroups + 1);
  int *d_res = reinterpret_cast<int *>(d_cand + (size_t)ngroups + 1);
  BTLE_CUDA_S(ctx, cudaMemsetAsync(d_in, 0, in_al, ctx->stream));
  BTLE_CUDA_S(ctx, cudaMemcpyAsync(d_in, rxp, valid, cudaMemcpyHostToDevice, ctx->stream));
  search_kernel<<<1, 128, 0, ctx->stream>>>(d_in, search_len, cfg, ngroups, d_pd, d_cand, d_res);
  BTLE_CUDA_S(ctx, cudaGetLastError());
  int res = -1;
  BTLE_CUDA_S(ctx, cudaMemcpyAsync(&res, d_res, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA_S(ctx, cudaStreamSynchronize(ctx->stream));
  return res;
#undef BTLE_CUDA_S
}

int btle_b200_demod_byte(btle_b200_ctx *ctx, const int8_t *rxp, int num_byte, uint8_t *out_byte) {
  if (!ctx || !rxp || !out_byte || num_byte < 0 || num_byte > 64) return BTLE_EINVAL;
  if (num_byte == 0) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t in_bytes = 64 * (size_t)num_byte - 4;       // last read index: 8*(8n-1)+3
  int rc = leaf_buf(ctx, 8192);
  if (rc) return rc;
  int8_t *d_in = static_cast<int8_t *>(ctx->d_leaf);
  uint8_t *d_o = reinterpret_cast<uint8_t *>(d_in) + 4608;
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_in, rxp, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
  demod_byte_kernel<<<1, 64, 0, ctx->stream>>>(d_in, num_byte, d_o);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaMemcpyAsync(out_byte, d_o, num_byte, cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

int btle_b200_scramble_byte(btle_b200_ctx *ctx, const uint8_t *byte_in, int num_byte, int channel, int table_offset,
                            uint8_t *byte_out) {
  if (!ctx || !byte_in || !byte_out || num_byte < 0 || channel < 0 || channel > 39 || table_offset < 0 ||
      table_offset + num_byte > 42)
    return BTLE_EINVAL;
  if (num_byte == 0) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc = leaf_buf(ctx, 256);
  if (rc) return rc;
  uint8_t *d_in = static_cast<uint8_t *>(ctx->d_leaf), *d_o = d_in + 64;
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_in, byte_in, num_byte, cudaMemcpyHostToDevice, ctx->stream));
  scramble_kernel<<<1, 64, 0, ctx->stream>>>(d_in, num_byte, channel, table_offset, d_o);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaMemcpyAsync(byte_out, d_o, num_byte, cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

int btle_b200_crc24_byte(btle_b200_ctx *ctx, const uint8_t *byte_in, int num_byte, uint32_t init_hex, uint32_t *crc_out) {
  if (!ctx || (!byte_in && num_byte) || !crc_out || num_byte < 0 || num_byte > 4096) return BTLE_EINVAL;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc = leaf_buf(ctx, 8192);
  if (rc) return rc;
  uint8_t *d_in = static_cast<uint8_t *>(ctx->d_leaf);
  uint32_t *d_o = reinterpret_cast<uint32_t *>(d_in + 4096);
  if (num_byte) BTLE_CUDA(ctx, cudaMemcpyAsync(d_in, byte_in, num_byte, cudaMemcpyHostToDevice, ctx->stream));
  crc24_kernel<<<1, 1, 0, ctx->stream>>>(d_in, num_byte, init_hex, d_o);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaMemcpyAsync(crc_out, d_o, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

uint32_t btle_b200_crc_init_reorder(uint32_t crc_init) { return crc_init_reorder(crc_init); }

int btle_b200_tx_modulate_device(btle_b200_ctx *ctx, const uint8_t *d_air, const int32_t *d_nbytes, size_t n_packets,
                                 size_t max_bytes, int sps, int8_t *d_out_i, int8_t *d_out_q, void *cuda_stream) {
  if (!ctx || !d_air || !d_nbytes || !d_out_i || (sps != 4 && sps != 8) || (sps == 8 && !d_out_q) || max_bytes == 0 ||
      max_bytes > 128 || n_packets > 0x7FFFFFFFu)
    return BTLE_EINVAL;
  if (n_packets == 0) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  if (sps == 4) tx_modulate_kernel<4><<<(unsigned)n_packets, 256, 0, st>>>(d_air, d_nbytes, (int)max_bytes, d_out_i, d_out_q);
  else tx_modulate_kernel<8><<<(unsigned)n_packets, 512, 0, st>>>(d_air, d_nbytes, (int)max_bytes, d_out_i, d_out_q);
  BTLE_CUDA(ctx, cudaGetLastError());
  return BTLE_OK;
}

int btle_b200_synth_streams_device(btle_b200_ctx *ctx, int8_t *d_iq, size_t n_streams, size_t stride, size_t n_int8,
                                   const btle_stream_cfg *cfgs, const btle_synth_cfg *sc, btle_synth_truth *d_truth,
                                   size_t truth_cap, size_t *n_slots_out, void *cuda_stream) {
  if (!ctx || !d_iq || !cfgs || !sc || n_streams == 0 || (n_streams > 1 && stride < n_int8)) return BTLE_EINVAL;
  if (sc->slot_samples < 1600 || sc->amplitude < 0 || sc->amplitude > 127 || sc->noise < 0 || sc->noise > 2 || sc->corrupt_every < 0 ||
      sc->straddle_every < 0 || (sc->straddle_every > 0 && (sc->straddle_every < 2 || sc->slot_samples < 3200))) {
    ctx->err = "synth: slot_samples >= 1600 (>= 3200 and straddle_every >= 2 with straddling), amplitude 0..127, noise 0..2";
    return BTLE_EINVAL;
  }
  int rc = validate_cfgs(ctx, cfgs, n_streams);
  if (rc) return rc;
  const size_t n_slots = (n_int8 / 2) / (size_t)sc->slot_samples;
  if (n_slots_out) *n_slots_out = n_slots;
  if (d_truth && truth_cap < n_slots * n_streams) { ctx->err = "synth: truth buffer too small"; return BTLE_EINVAL; }
  if (n_slots * n_streams > 0x7FFFFFFFull) { ctx->err = "synth: too many slots for one launch"; return BTLE_EINVAL; }
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  CfgSlot *cs = nullptr;
  rc = upload_cfgs(ctx, cfgs, n_streams, st, &cs);
  if (rc) return rc;
  synth_noise_kernel<<<ctx->num_sms * 8, 256, 0, st>>>(d_iq, (long long)stride, (long long)n_int8, (int)n_streams, sc->seed, sc->noise);
  BTLE_CUDA(ctx, cudaGetLastError());
  if (n_slots && sc->amplitude > 0) {
    synth_bursts_kernel<<<(unsigned)(n_slots * n_streams), 256, 0, st>>>(d_iq, (long long)stride, (long long)n_int8, cs->d, *sc,
                                                                          (long long)n_slots, d_truth);
    BTLE_CUDA(ctx, cudaGetLastError());
  }
  BTLE_CUDA(ctx, cudaEventRecord(cs->last_use, st));
  return BTLE_OK;
}

int btle_b200_model_rx_batch_device(btle_b200_ctx *ctx, const int16_t *d_i, const int16_t *d_q, size_t n_packets,
                                    size_t n_samples, int sps, int channel, uint32_t crc_init, uint32_t access_addr,
                                    btle_model_rx_rec *d_out, void *cuda_stream) {
  if (!ctx || !d_i || !d_q || !d_out || sps < 1 || sps > 64 || channel < 0 || channel > 39 || n_samples % (size_t)sps ||
      n_samples / (size_t)sps < 34 || n_samples / (size_t)sps > 32u * kModelMaxWords || n_packets > 0x7FFFFFFFu / 4 * 4)
    return BTLE_EINVAL;
  if (n_packets == 0) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  const int adv = (channel >= 37 && channel <= 39);
  model_rx_batch_kernel<<<(unsigned)((n_packets + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(cuda_stream)>>>(
      d_i, d_q, 1, nullptr, (int)n_packets, (int)n_samples, sps, adv, channel, access_addr, crc_init_reorder(crc_init), d_out);
  BTLE_CUDA(ctx, cudaGetLastError());
  return BTLE_OK;
}

int btle_b200_model_rx_batch(btle_b200_ctx *ctx, const int16_t *i, const int16_t *q, size_t n_packets, size_t n_samples,
                             int sps, int channel, uint32_t crc_init, uint32_t access_addr, btle_model_rx_rec *out) {
  if (!ctx || !i || !q || !out) return BTLE_EINVAL;
  if (n_packets == 0) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t nb = n_packets * n_samples * 2, a = (nb + 255) & ~size_t(255);
  int rc = leaf_buf(ctx, 2 * a + n_packets * sizeof(btle_model_rx_rec) + 256);
  if (rc) return rc;
  uint8_t *base = static_cast<uint8_t *>(ctx->d_leaf);
  int16_t *d_i = reinterpret_cast<int16_t *>(base), *d_q = reinterpret_cast<int16_t *>(base + a);
  btle_model_rx_rec *d_o = reinterpret_cast<btle_model_rx_rec *>(base + 2 * a);
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_i, i, nb, cudaMemcpyHostToDevice, ctx->stream));
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_q, q, nb, cudaMemcpyHostToDevice, ctx->stream));
  rc = btle_b200_model_rx_batch_device(ctx, d_i, d_q, n_packets, n_samples, sps, channel, crc_init, access_addr, d_o, ctx->stream);
  if (rc) return rc;
  BTLE_CUDA(ctx, cudaMemcpyAsync(out, d_o, n_packets * sizeof(btle_model_rx_rec), cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

int btle_b200_sps8_hits_device(btle_b200_ctx *ctx, const int16_t *d_iq16, size_t n_samples, uint32_t access_addr, int64_t *d_hits, size_t cap,
                               uint32_t *d_count, void *cuda_stream) {
  if (!ctx || !d_iq16 || !d_count || (!d_hits && cap) || (reinterpret_cast<uintptr_t>(d_iq16) & 3)) return BTLE_EINVAL;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  BTLE_CUDA(ctx, cudaMemsetAsync(d_count, 0, sizeof(unsigned), st));
  if (!n_samples) return BTLE_OK;
  int rc = launch_sps8_hits(ctx, d_iq16, n_samples, access_addr, reinterpret_cast<long long *>(d_hits), std::min<size_t>(cap, 0xFFFFFFFFu), d_count, st);
  if (rc) return rc;
  BTLE_CUDA(ctx, cudaGetLastError());
  ctx->last_launches = 1;
  return BTLE_OK;
}

// Streaming form of the Python model's receiver over an 8-Msps interleaved int16 capture (see include/btle_b200.h).
int btle_b200_rx_sps8(btle_b200_ctx *ctx, const int16_t *iq16, size_t n_samples, int channel, uint32_t crc_init, uint32_t access_addr,
                      btle_sps8_rec *out, size_t cap, size_t *n_out) {
  if (!ctx || (!iq16 && n_samples) || !n_out || (!out && cap) || channel < 0 || channel > 39) return BTLE_EINVAL;
  *n_out = 0;
  if (n_samples < (size_t)BTLE_SPS8_WINDOW) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t bytes = n_samples * 4, hit_cap = n_samples / 256 + 4096;
  int rc = ensure(ctx, reinterpret_cast<void **>(&ctx->d_iq), &ctx->d_iq_bytes, bytes + 256);
  if (rc) return rc;
  rc = leaf_buf(ctx, hit_cap * 8 + 256);
  if (rc) return rc;
  long long *d_hits = static_cast<long long *>(ctx->d_leaf);
  const int16_t *d_iq = reinterpret_cast<const int16_t *>(ctx->d_iq);
  rc = h2d_rows(ctx, ctx->d_iq, bytes, reinterpret_cast<const int8_t *>(iq16), bytes, bytes, 1, st);
  if (rc) return rc;
  BTLE_CUDA(ctx, cudaMemsetAsync(ctx->d_count, 0, sizeof(unsigned), st));
  rc = launch_sps8_hits(ctx, d_iq, n_samples, access_addr, d_hits, hit_cap, ctx->d_count, st);
  if (rc) return rc;
  BTLE_CUDA(ctx, cudaMemcpyAsync(ctx->h_count, ctx->d_count, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  BTLE_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_launches = 1;
  size_t n_hits = *ctx->h_count;
  if (n_hits > hit_cap) { ctx->err = "rx_sps8: more access-address hits than the hit buffer holds"; return BTLE_EOVERFLOW; }
  if (!n_hits) return BTLE_OK;
  std::vector<long long> hits(n_hits);
  BTLE_CUDA(ctx, cudaMemcpyAsync(hits.data(), d_hits, n_hits * 8, cudaMemcpyDeviceToHost, st));
  BTLE_CUDA(ctx, cudaStreamSynchronize(st));
  std::sort(hits.begin(), hits.end());
  // candidates: the first hit of every cluster (hits closer than the shortest possible packet belong to one packet: the same
  // access address seen on neighbouring sample phases), with its window
  std::vector<long long> cand, win;
  long long last = -(1ll << 60);
  for (long long h : hits) {
    if (h < last + 8ll * BTLE_SPS8_MIN_PACKET_SYMBOLS) continue;
    last = h;
    long long w0 = 8 * (h / 8 - BTLE_SPS8_MARGIN_SYMBOLS);
    if (w0 < 0) w0 = 0;
    if (w0 + BTLE_SPS8_WINDOW > (long long)n_samples) continue;             // the window must lie inside the capture
    cand.push_back(h);
    win.push_back(w0);
  }
  if (cand.empty()) return BTLE_OK;
  const size_t nc = cand.size();
  rc = leaf_buf(ctx, nc * 8 + nc * sizeof(btle_model_rx_rec) + 512);
  if (rc) return rc;
  long long *d_win = static_cast<long long *>(ctx->d_leaf);
  btle_model_rx_rec *d_rec = reinterpret_cast<btle_model_rx_rec *>(reinterpret_cast<uint8_t *>(ctx->d_leaf) + ((nc * 8 + 255) & ~size_t(255)));
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_win, win.data(), nc * 8, cudaMemcpyHostToDevice, st));
  const int adv = (channel >= 37 && channel <= 39);
  model_rx_batch_kernel<<<(unsigned)((nc + 3) / 4), 128, 0, st>>>(d_iq, d_iq + 1, 2, d_win, (int)nc, BTLE_SPS8_WINDOW, 8, adv, channel, access_addr,
                                                                  crc_init_reorder(crc_init), d_rec);
  BTLE_CUDA(ctx, cudaGetLastError());
  std::vector<btle_model_rx_rec> recs(nc);
  BTLE_CUDA(ctx, cudaMemcpyAsync(recs.data(), d_rec, nc * sizeof(btle_model_rx_rec), cudaMemcpyDeviceToHost, st));
  BTLE_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_launches = 2;
  // greedy: a candidate inside the packet accepted before it is part of that packet
  long long cursor = -1;
  size_t n = 0;
  for (size_t k = 0; k < nc; ++k) {
    if (cand[k] < cursor) continue;
    const btle_model_rx_rec &r = recs[k];
    long long at = cand[k];
    if (r.found) at = win[k] + 8ll * r.start + (r.crc_ok ? r.phase : r.found - 1);
    const int plen = r.found ? r.payload_len : 0;
    cursor = at + 8ll * (32 + 16 + 8 * plen + 24);
    if (n < cap) { out[n].sample = at; out[n].window = win[k]; out[n].rx = r; }
    ++n;
  }
  *n_out = n;
  if (n > cap) { ctx->err = "output capacity too small"; return BTLE_EOVERFLOW; }
  return BTLE_OK;
}

int btle_b200_ber_run(btle_b200_ctx *ctx, const btle_ber_cfg *cfg, size_t n_packets, btle_ber_result *out) {
  if (!ctx || !cfg || !out || cfg->channel < 0 || cfg->channel > 39) return BTLE_EINVAL;
  memset(out, 0, sizeof *out);
  if (!n_packets) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t B = std::min<size_t>(n_packets, 32768);
  const size_t iq_bytes = B * kBerSamples * sizeof(int16_t);
  const size_t a_iq = (iq_bytes + 255) & ~size_t(255), a_tr = (B * 40 + 255) & ~size_t(255), a_rec = (B * sizeof(btle_model_rx_rec) + 255) & ~size_t(255);
  int rc = leaf_buf(ctx, 2 * a_iq + a_tr + a_rec + 256);
  if (rc) return rc;
  uint8_t *base = static_cast<uint8_t *>(ctx->d_leaf);
  int16_t *d_i = reinterpret_cast<int16_t *>(base), *d_q = reinterpret_cast<int16_t *>(base + a_iq);
  uint8_t *d_truth = base + 2 * a_iq;
  btle_model_rx_rec *d_rec = reinterpret_cast<btle_model_rx_rec *>(base + 2 * a_iq + a_tr);
  unsigned long long *d_acc = reinterpret_cast<unsigned long long *>(base + 2 * a_iq + a_tr + a_rec);
  BTLE_CUDA(ctx, cudaMemsetAsync(d_acc, 0, 3 * sizeof(unsigned long long), st));
  cudaEvent_t e0, e1;
  BTLE_CUDA(ctx, cudaEventCreate(&e0));
  BTLE_CUDA(ctx, cudaEventCreate(&e1));
  BTLE_CUDA(ctx, cudaEventRecord(e0, st));
  const int adv = (cfg->channel >= 37);
  int launches = 0;
  for (size_t done = 0; done < n_packets; done += B) {
    const int n = (int)std::min(B, n_packets - done);
    ber_synth_kernel<<<n, 384, 0, st>>>(*cfg, (unsigned long long)done, n, d_i, d_q, d_truth);
    model_rx_batch_kernel<<<(n + 3) / 4, 128, 0, st>>>(d_i, d_q, 1, nullptr, n, kBerSamples, 8, adv, cfg->channel, cfg->access_addr,
                                                      crc_init_reorder(cfg->crc_init), d_rec);
    ber_score_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_rec, d_truth, n, d_acc);
    launches += 3;
  }
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaEventRecord(e1, st));
  unsigned long long acc[3];
  BTLE_CUDA(ctx, cudaMemcpyAsync(acc, d_acc, sizeof acc, cudaMemcpyDeviceToHost, st));
  BTLE_CUDA(ctx, cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  out->packets = n_packets; out->pkt_err = acc[0]; out->bit_err = acc[1]; out->aa_miss = acc[2];
  out->bit_total = (uint64_t)n_packets * 8 * kBerPduBytes;
  out->seconds = ms * 1e-3;
  ctx->last_launches = launches;
  return BTLE_OK;
}

int btle_b200_gfsk_demod_i16(btle_b200_ctx *ctx, const int16_t *i, const int16_t *q, size_t n, int8_t *bit_out,
                             int32_t *signal_out) {
  if (!ctx || !i || !q || !bit_out || !signal_out) return BTLE_EINVAL;
  if (n < 2) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t a = (2 * n + 255) & ~size_t(255);
  int rc = leaf_buf(ctx, 2 * a + 4 * n + n + 512);
  if (rc) return rc;
  uint8_t *base = static_cast<uint8_t *>(ctx->d_leaf);
  int16_t *d_i = reinterpret_cast<int16_t *>(base), *d_q = reinterpret_cast<int16_t *>(base + a);
  int32_t *d_s = reinterpret_cast<int32_t *>(base + 2 * a);
  int8_t *d_b = reinterpret_cast<int8_t *>(base + 2 * a + 4 * n);
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_i, i, 2 * n, cudaMemcpyHostToDevice, ctx->stream));
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_q, q, 2 * n, cudaMemcpyHostToDevice, ctx->stream));
  gfsk_demod_i16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_i, d_q, (long long)n, d_b, d_s);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaMemcpyAsync(bit_out, d_b, n - 1, cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaMemcpyAsync(signal_out, d_s, 4 * (n - 1), cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

long btle_b200_search_bit_sequence(btle_b200_ctx *ctx, const int8_t *bit, size_t n, const int8_t *seq, size_t m) {
  if (!ctx || !bit || !seq || m == 0 || m > 4096) return BTLE_EINVAL - 1;     // -2: errors never collide with "-1 = not found"
  if (n < m) return -1;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return BTLE_ECUDA - 1;
  const size_t a = (n + 255) & ~size_t(255);
  if (leaf_buf(ctx, a + m + 512)) return BTLE_ENOMEM - 1;
  int8_t *d_b = static_cast<int8_t *>(ctx->d_leaf), *d_s = d_b + a;
  long long *d_first = reinterpret_cast<long long *>(d_b + a + ((m + 255) & ~size_t(255)));
  long long first = -1;                                     // all ones == "none" for the unsigned atomicMin
  cudaMemcpyAsync(d_b, bit, n, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(d_s, seq, m, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(d_first, &first, 8, cudaMemcpyHostToDevice, ctx->stream);
  search_seq_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_b, (long long)n, d_s, (int)m, d_first);
  cudaMemcpyAsync(&first, d_first, 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) { ctx->err = cudaGetErrorString(cudaGetLastError()); return BTLE_ECUDA - 1; }
  return (long)first;
}

int btle_b200_crc24_bits(btle_b200_ctx *ctx, const int8_t *bit_in, size_t n, const int8_t *state_init_bit, int8_t *crc_bits_out) {
  if (!ctx || (!bit_in && n) || !state_init_bit || !crc_bits_out) return BTLE_EINVAL;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t a = (n + 255) & ~size_t(255);
  int rc = leaf_buf(ctx, a + 512);
  if (rc) return rc;
  int8_t *d_b = static_cast<int8_t *>(ctx->d_leaf), *d_i = d_b + a, *d_o = d_b + a + 64;
  if (n) BTLE_CUDA(ctx, cudaMemcpyAsync(d_b, bit_in, n, cudaMemcpyHostToDevice, ctx->stream));
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_i, state_init_bit, 24, cudaMemcpyHostToDevice, ctx->stream));
  crc24_bits_kernel<<<1, 1, 0, ctx->stream>>>(d_b, (long long)n, d_i, d_o);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaMemcpyAsync(crc_bits_out, d_o, 24, cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

int btle_b200_scramble_bits(btle_b200_ctx *ctx, const int8_t *bit_in, size_t n, int channel, int8_t *bit_out) {
  if (!ctx || (!bit_in && n) || (!bit_out && n) || channel < 0 || channel > 63) return BTLE_EINVAL;
  if (n == 0) return BTLE_OK;
  BTLE_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t a = (n + 255) & ~size_t(255);
  int rc = leaf_buf(ctx, 2 * a);
  if (rc) return rc;
  int8_t *d_b = static_cast<int8_t *>(ctx->d_leaf), *d_o = d_b + a;
  BTLE_CUDA(ctx, cudaMemcpyAsync(d_b, bit_in, n, cudaMemcpyHostToDevice, ctx->stream));
  scramble_bits_kernel<<<1, 1, 0, ctx->stream>>>(d_b, (long long)n, channel, d_o);
  BTLE_CUDA(ctx, cudaGetLastError());
  BTLE_CUDA(ctx, cudaMemcpyAsync(bit_out, d_o, n, cudaMemcpyDeviceToHost, ctx->stream));
  BTLE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BTLE_OK;
}

void btle_b200_parse_adv_pdu_header_byte(const uint8_t *b, int *pdu_type, int *tx_add, int *rx_add, int *payload_len) {
  *pdu_type = b[0] & 0x0F;             // btle_rx.c:1950
  *tx_add = (b[0] & 0x40) != 0;        // :1955
  *rx_add = (b[0] & 0x80) != 0;        // :1959
  *payload_len = b[1] & 0x3F;          // :1962
}

void btle_b200_parse_ll_pdu_header_byte(const uint8_t *b, int *llid, int *nesn, int *sn, int *md, int *payload_len) {
  *llid = b[0] & 0x03;                 // btle_rx.c:1940
  *nesn = (b[0] & 0x04) != 0;
  *sn = (b[0] & 0x08) != 0;
  *md = (b[0] & 0x10) != 0;
  *payload_len = b[1] & 0x1F;          // :1944
}

}  // extern "C"
