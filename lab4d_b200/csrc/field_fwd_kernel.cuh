// Fused per-ray-sample forward of one Lab4D field (training-mode query_field) for sm_100a:
// TWO 128-sample tiles in flight per CTA.
//
// Persistent kernel, one CTA per SM, CTAs paired in clusters of 2 that share every weight chunk through
// TMA multicast.  Warp roles (384 threads, three warpgroups; setmaxnreg gives the two compute warpgroups 208 registers):
//   warps 0-3 : tile group 0, warps 4-7 : tile group 1.  One thread per sample (thread = tile row = TMEM lane):
//               sample placement, camera -> field, dual-quaternion blend skinning (+ DenseWarp), Fourier embedding
//               into swizzled shared memory, and every layer's epilogue straight out of TMEM.
//   warp 8    : TMA producer - streams pre-packed weight chunks (cp.async.bulk, multicast to both CTAs of the
//               cluster) through a 3-slot ring of 32 KB, in the order [block b, group 0][block b, group 1][block b+1, ...
//               (a block = one GEMM or one N-half of a 256-wide layer).
//   warps 9-10: tcgen05.mma issuers, one per tile group (one elected lane each; warp 9 owns the TMEM allocation).  Each
//               walks the MmaBlock list of program.h out of the kernel parameters - every descriptor stays in uniform
//               registers - and consumes its own group's ring slots: while one group runs an epilogue or its SIMT
//               geometry, the tensor pipe works on the other group's tile, so the round-trip latencies of the 40-odd
//               dependent GEMMs of a tile overlap.  Full barriers are per (group, slot): each is waited on by exactly
//               one issuer, phase after phase (a shared barrier would alias parities between the groups).
//   warp 11   : idle (register donor).
// Other entries reuse the kernel with a shorter block list: b200r_points_fwd (NeRF.forward on given points) and
// b200r_warp_fwd (one warp of given points); b200r_ray_batch.depth replaces the uniform sample placement.
// TMEM (512 columns): per group 128 fp32 accumulator columns + 128 columns holding 256 16-bit activations.  All
// hidden activations live in TMEM and feed the next layer as the A operand (TS form); the 256-wide layers run as
// two N-halves on the same accumulator: the epilogue of half 0 drains it into registers while half 1 is being
// multiplied, and both halves are written back in place once the layer's MMAs have read their input.
// Shared memory holds only the embedding operand chunks (2 x 16 KB per group), the weight ring, the constant
// block and one per-frame block per group.  HBM sees O(100 B) per sample of outputs.
//
// Restates (not ports) lab4d/nnutils/{nerf,deformable,feature,warping,skinning,embedding,visibility}.py
// and lab4d/utils/{render_utils,geom_utils,quat_transform}.py - see include/b200r.h for file:line.
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include <type_traits>

#include "kernels.h"
#include "ptx.cuh"

#ifndef B200R_CLUSTER
#define B200R_CLUSTER 2
#endif

namespace b200r {
namespace fwd {

constexpr int kCluster = B200R_CLUSTER;
constexpr int kNumStages = 3;
constexpr int kGroups = 2;
constexpr int kGroupThreads = 128;
constexpr int kComputeThreads = kGroups * kGroupThreads;
constexpr int kThreads = kComputeThreads + 128;  // warpgroup 2 = producer warp, MMA warp, two idle warps (register donors)
constexpr int kRegsCompute = 208, kRegsAux = 88;        // setmaxnreg: 2 x 128 x 208 + 128 x 88 = 64512 <= 65536
constexpr int kArenaGroup = 2 * kAChunkBytes;           // CH_PE, CH_EXTRA
constexpr int kSmemArena = kGroups * kArenaGroup;        // 64 KB
constexpr int kSmemRing = kNumStages * kWStageBytes;     // 96 KB
constexpr int kTmemAcc = 0, kTmemAct = 256, kTmemGroup = 128;
constexpr int kBarBytes = 256;                            // mbarriers + TMEM slot
constexpr int kSdfPartBytes = 2 * 4 * kTileRows * 4;      // SPLIT: 8 partial sdf sums per row

struct Q4 { float w, x, y, z; };
__device__ __forceinline__ Q4 qmul(const Q4& a, const Q4& b) {
  return {a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z, a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
          a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x, a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w};
}
__device__ __forceinline__ Q4 qconj(const Q4& a) { return {a.w, -a.x, -a.y, -a.z}; }
__device__ __forceinline__ float3 qrot(const Q4& q, const float3& p) {  // quaternion_apply
  Q4 t = qmul(q, Q4{0.f, p.x, p.y, p.z});
  Q4 r = qmul(t, qconj(q));
  return make_float3(r.x, r.y, r.z);
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint4 lds128u(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds32u(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts16(uint32_t a, uint16_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"(v) : "memory"); }

template <int V>
using IC = std::integral_constant<int, V>;

// SPLIT (operand_dtype 2, "fp16x3"): every MMA operand is carried as an fp16 head plus the fp16 tail of its rounding
// error and every product as head*head + tail*head + head*tail (fp32 accumulate): ~22-bit operands, the parity mode that
// meets the 1e-4 rendered-RGB contract.  The tails take the TMEM / shared-memory space of tile group 1, so a CTA then
// keeps ONE tile in flight: activation tails in columns [384, 512), embedding tails in group 1's arena chunks.  Both
// groups' warps work on that tile: warps q and 4+q read the same TMEM lane quadrant and split every epilogue's 32-column
// blocks (group g takes the blocks [g * nb / 2, (g + 1) * nb / 2) of each N-half), so every c2m barrier counts 8 warps.
// Per-row scalar work (sample placement, skinning blend, embedding, heads, per-sample outputs) stays on group 0.
// Columns [128, 256) are the accumulator of a wide layer's N-half 1, whose MMAs then overlap the epilogue of half 0.
// SAVE (training forward, b200r_field_fwd with a tape): every epilogue also records the 16-bit operand it produced in the
// tape's chunk image and one word of ReLU sign bits per 32 columns (program.h TapeLayout) for the backward kernels.
template <class Op, int B, int LMAX, bool DENSE, int WIDTH, bool SPLIT, bool SAVE>
__global__ void __launch_bounds__(kThreads, 1) field_fwd_kernel(const __grid_constant__ FieldKernelParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* arena = smem;
  uint8_t* ring = smem + kSmemArena;
  float* cblk = reinterpret_cast<float*>(ring + kSmemRing);
  float* fblk = cblk + p.prog.cl.n_floats;  // one frame block per tile group
  uint64_t* bars = reinterpret_cast<uint64_t*>(fblk + kGroups * p.prog.fl.n_floats);
  // full barriers are per (group, stage): every barrier is then waited on by exactly one issuer, phase after phase,
  // so a parity wait can never alias with a fill that belongs to the other group's use of the same stage
  uint64_t* full_bar = bars;                  // [group][kNumStages]
  uint64_t* empty_bar = bars + 2 * kNumStages;  // [kNumStages]
  uint64_t* c2m = bars + 3 * kNumStages;      // [group][4] compute warps -> MMA thread, indexed by BAR_*
  uint64_t* m2c = bars + 3 * kNumStages + 8;  // [group][4] MMA thread (tcgen05.commit) -> compute warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kNumStages + 16);
  // SPLIT: MODE 1 partial sdf dot products, [2 * (WIDTH / 64) blocks][128 rows], summed by group 0 in block order
  const uint32_t sdf_part_s = smem_u32(bars) + kBarBytes;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
  if (threadIdx.x == 0) {
    for (int i = 0; i < kNumStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&full_bar[kNumStages + i], 1); mbar_init(&empty_bar[i], kCluster); }
    // one arrival per warp working on the group's tile (SPLIT: both groups' warps)
    for (int i = 0; i < 8; ++i) { mbar_init(&c2m[i], SPLIT ? 8 : 4); mbar_init(&m2c[i], 1); }
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();  // peer barriers are initialised before any multicast can land
  tc_fence_after_sync();
  if (*tmem_slot != 0) __trap();        // the CTA allocates all 512 columns, so the allocation starts at column 0
  constexpr uint32_t tmem_base = 0;
  const Program& P = p.prog;
  constexpr int kActive = SPLIT ? 1 : kGroups;  // tile groups in flight
  const int pair_stride = kActive * (int)gridDim.x;
  const int iters = (p.n_tiles + pair_stride - 1) / pair_stride;  // identical in both CTAs of a cluster
  const uint32_t cta_rank = kCluster > 1 ? cluster_ctarank() : 0;
  const uint16_t cmask = (uint16_t)((1u << kCluster) - 1);

  if (warp >= 8) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsAux));
  if (warp == 8) {
    // =============================================================== TMA producer
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int it = 0; it < iters; ++it) {
        int st = 0;
        while (st < P.n_steps) {
          int end = st;
          while (P.steps[end].commit == 0) ++end;
          ++end;
          for (int g = 0; g < kActive; ++g) {
            for (int s = st; s < end; ++s) {
              const MmaStep& S = P.steps[s];
              const uint32_t bytes = (uint32_t)S.n * 128u * S.n_sub;
              const uint32_t part = bytes / kCluster;
              uint64_t* fb = &full_bar[g * kNumStages + stage];
              mbar_wait(&empty_bar[stage], phase ^ 1);  // both CTAs' MMAs are done with this slot
              mbar_arrive_expect_tx(fb, bytes);
              const uint8_t* src = p.packed + S.w_off + cta_rank * part;
              uint8_t* dst = ring + stage * kWStageBytes + cta_rank * part;
              if (kCluster > 1) tma_bulk_g2s_mcast(dst, src, part, fb, cmask);
              else tma_bulk_g2s(dst, src, part, fb);
              if (++stage == kNumStages) { stage = 0; phase ^= 1; }
            }
          }
          st = end;
        }
      }
    }
  } else if (warp == 9 || (warp == 10 && !SPLIT)) {
    // =============================================================== MMA issuers: warp 9 -> tile group 0, warp 10 -> group 1.
    // Ring slots are filled in the global order [block b, group 0][block b, group 1][block b+1, group 0]...; each
    // issuer consumes its own group's slots (signalled on its own full barriers) and steps over the other's.  Everything here is warp-uniform and comes
    // from the kernel parameters (MmaBlock), so descriptors and addresses stay in uniform registers.
    const int g = warp - 9;
    uint32_t stage = 0;
    uint32_t full_par = 0;   // bit s = parity of this group's full barrier of stage s
    uint32_t bar_phase = 0;  // bit i = parity of c2m[g][i]
    uint64_t* full_g = full_bar + g * kNumStages;
    const uint32_t desc_hi = (uint32_t)(umma_desc_k_sw128(0) >> 32);
    const uint32_t bd_lo0 = (uint32_t)umma_desc_k_sw128(smem_u32(ring));
    const uint32_t ad_lo0 = (uint32_t)umma_desc_k_sw128(smem_u32(arena)) + (uint32_t)g * (kArenaGroup >> 4);
    const uint32_t d = kTmemAcc + kTmemGroup * g;      // TMEM base is 0 (checked above): the CTA owns all 512 columns
    const uint32_t act0 = kTmemAct + kTmemGroup * g;
    uint64_t* c2m_g = c2m + 4 * g;
    uint64_t* m2c_g = m2c + 4 * g;
    auto mk = [&](uint32_t lo) { return ((uint64_t)desc_hi << 32) | lo; };
    auto advance = [&]() { if (++stage == kNumStages) stage = 0; };
    auto wait_full = [&]() {
      mbar_wait(&full_g[stage], (full_par >> stage) & 1u);
      full_par ^= 1u << stage;
      tc_fence_after_sync();
    };
    auto skip = [&](uint32_t cnt) {  // step over the other group's slots (they have their own full barriers)
      for (uint32_t j = 0; j < cnt; ++j) advance();
    };
    auto release = [&]() {  // frees the ring slot (in both CTAs) once the MMAs issued so far have read it
      if (kCluster > 1) umma_commit_mcast(&empty_bar[stage], cmask);
      else umma_commit(&empty_bar[stage]);
    };
    const int n_blocks = P.n_blocks;
    for (int it = 0; it < iters; ++it) {
#pragma unroll 1
      for (int b = 0; b < n_blocks; ++b) {
        const MmaBlock& Bk = P.blocks[b];
        const uint32_t n = (uint32_t)Bk.n16 << 4, ss = Bk.ss, ts_slots = Bk.ts_slots, cnt = (ss ? 1u : 0u) + ts_slots;
        const uint32_t idesc = umma_idesc_f16(Op::kFmt, 0) | ((n >> 3) << 17);
        const uint32_t tile2 = n << 3;  // descriptor offset of a slot's second weight tile (n rows x 128 B)
        if (g == 1) skip(cnt);
        const uint32_t wt = Bk.wait, cm = Bk.commit;
        // SPLIT: N-half 1 of a wide layer (the block that waits on BAR_H0) accumulates into columns [128, 256), so it
        // need not wait for the epilogue to drain half 0
        const bool half1 = SPLIT && wt == BAR_H0;
        if (wt && !half1) {
          mbar_wait(&c2m_g[wt], (bar_phase >> wt) & 1u);
          bar_phase ^= 1u << wt;
        }
        uint32_t acc = 0;
        if constexpr (SPLIT) {
          // one ring slot per K chunk: [head tile][tail tile]; operand tails: embedding chunks of group 1's arena,
          // activation columns + kTmemGroup.  D += Ah Wh + Al Wh + Ah Wl per k-step.
          const uint32_t dd = half1 ? d + kTmemGroup : d;
          const uint32_t ks_ss[2] = {ss & 7u, (ss >> 3) & 7u};
          const uint32_t n_ss = ss ? (ks_ss[1] ? 2u : 1u) : 0u;
          for (uint32_t c = 0; c < n_ss; ++c) {
            wait_full();
            const uint32_t bd = bd_lo0 + stage * (kWStageBytes >> 4), bl = bd + tile2;
            const bool last = c + 1 == n_ss && ts_slots == 0;
            if (elect_one()) {
              const uint32_t ah = ad_lo0 + (uint32_t)((Bk.ss_chunks >> (4 * c)) & 15) * (kAChunkBytes >> 4), al = ah + (kArenaGroup >> 4);
              for (uint32_t k = 0; k < ks_ss[c]; ++k) {
                umma_f16_ss(dd, mk(ah + 2 * k), mk(bd + 2 * k), idesc, acc | k);
                umma_f16_ss(dd, mk(al + 2 * k), mk(bd + 2 * k), idesc, 1u);
                umma_f16_ss(dd, mk(ah + 2 * k), mk(bl + 2 * k), idesc, 1u);
              }
              release();
              if (last && cm) umma_commit(&m2c_g[cm]);
            }
            __syncwarp();
            advance();
            acc = 1;
          }
          uint32_t a = act0;
#pragma unroll 1
          for (uint32_t j = 0; j < ts_slots; ++j) {
            wait_full();
            const uint32_t bd = bd_lo0 + stage * (kWStageBytes >> 4), bl = bd + tile2;
            const bool last = j + 1 == ts_slots;
            const uint32_t ks = last ? (uint32_t)Bk.ts_ks2_last : 4u;
            if (elect_one()) {
              for (uint32_t k = 0; k < ks; ++k) {
                umma_f16_ts(dd, a + 8 * k, mk(bd + 2 * k), idesc, acc | k);
                umma_f16_ts(dd, a + kTmemGroup + 8 * k, mk(bd + 2 * k), idesc, 1u);
                umma_f16_ts(dd, a + 8 * k, mk(bl + 2 * k), idesc, 1u);
              }
              release();
              if (last && cm) umma_commit(&m2c_g[cm]);
            }
            __syncwarp();
            advance();
            acc = 1;
            a += 32;
          }
          continue;
        }
        if (ss) {  // embedding chunk(s) from shared memory
          wait_full();
          const uint32_t bd = bd_lo0 + stage * (kWStageBytes >> 4);
          if (elect_one()) {
            const uint32_t ks = ss & 7u, ks2 = (ss >> 3) & 7u;
            const uint32_t a0 = ad_lo0 + (uint32_t)(Bk.ss_chunks & 15) * (kAChunkBytes >> 4);
            const uint32_t a1 = ad_lo0 + (uint32_t)(Bk.ss_chunks >> 4) * (kAChunkBytes >> 4);
            for (uint32_t k = 0; k < ks; ++k) umma_f16_ss(d, mk(a0 + 2 * k), mk(bd + 2 * k), idesc, k ? 1u : 0u);
            for (uint32_t k = 0; k < ks2; ++k) umma_f16_ss(d, mk(a1 + 2 * k), mk(bd + tile2 + 2 * k), idesc, 1u);
            release();
            if (cm && ts_slots == 0) umma_commit(&m2c_g[cm]);
          }
          __syncwarp();
          advance();
          acc = 1;
        }
        uint32_t a = act0;
#pragma unroll 1
        for (uint32_t j = 0; j < ts_slots; ++j) {  // activations from TMEM, 64 columns (128 values) per slot
          wait_full();
          const uint32_t bd = bd_lo0 + stage * (kWStageBytes >> 4), bd2 = bd + tile2;
          const bool last = j + 1 == ts_slots;
          if (elect_one()) {
            umma_f16_ts(d, a, mk(bd), idesc, acc);
            umma_f16_ts(d, a + 8, mk(bd + 2), idesc, 1u);
            umma_f16_ts(d, a + 16, mk(bd + 4), idesc, 1u);
            umma_f16_ts(d, a + 24, mk(bd + 6), idesc, 1u);
            if (!last || Bk.ts_ks2_last == 4) {
              umma_f16_ts(d, a + 32, mk(bd2), idesc, 1u);
              umma_f16_ts(d, a + 40, mk(bd2 + 2), idesc, 1u);
              umma_f16_ts(d, a + 48, mk(bd2 + 4), idesc, 1u);
              umma_f16_ts(d, a + 56, mk(bd2 + 6), idesc, 1u);
            } else {
              for (uint32_t k = 0; k < Bk.ts_ks2_last; ++k) umma_f16_ts(d, a + 32 + 8 * k, mk(bd2 + 2 * k), idesc, 1u);
            }
            release();
            if (last && cm) umma_commit(&m2c_g[cm]);
          }
          __syncwarp();
          advance();
          acc = 1;
          a += 64;
        }
        if (g == 0) skip(cnt);
      }
    }
  }
  } else {
    // =============================================================== compute / epilogue warps
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsCompute));
    const int g = warp >> 2, q = warp & 3;
    // SPLIT: both groups work on group 0's tile (its TMEM, arena, frame block, scratch and barriers); group g then only
    // selects the column blocks of an epilogue, and group 0 alone does the per-row scalar work (`lead`)
    const int tg = SPLIT ? 0 : g;
    const bool lead = !SPLIT || g == 0;
    constexpr int kTileThreads = SPLIT ? kComputeThreads : kGroupThreads;  // threads working on one tile
    const int gtid = threadIdx.x & (kGroupThreads - 1);
    const int ttid = SPLIT ? (int)threadIdx.x : gtid;
    const uint32_t row = (uint32_t)(q * 32 + lane);  // tile row == TMEM lane
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t tD = t_lane + kTmemAcc + kTmemGroup * tg;  // this tile's accumulator
    const uint32_t tA = t_lane + kTmemAct + kTmemGroup * tg;  // this tile's 16-bit activations (2 per column)
    constexpr uint32_t kTail = kTmemGroup;                      // SPLIT: activation tails live in group 1's columns
    uint64_t* c2m_g = c2m + 4 * tg;
    uint64_t* m2c_g = m2c + 4 * tg;
    uint32_t all_phase = 0, half_phase = 0;
    constexpr int HN = WIDTH / 2, NBLK = HN / 32;  // N-half of the wide layers; 32-column blocks per half
    const int lid_delta = 0, lid_vis = B > 0 ? 3 : 0, lid_base = lid_vis + 2, lid_rgb0 = lid_base + p.desc.D + 1,
              lid_color = lid_rgb0 + 1, lid_feat = lid_color + 3, lid_dense = lid_feat + (p.desc.has_feature ? 6 : 0);
    const ConstLayout& CL = P.cl;
    const FrameLayout& FL = P.fl;
    float* fblk_g = fblk + tg * FL.n_floats;
    const uint32_t cblk_s = smem_u32(cblk), fblk_s = smem_u32(fblk_g);
    const uint32_t pe_s = smem_u32(arena) + tg * kArenaGroup, extra_s = pe_s + kAChunkBytes;
    const uint32_t rowx = row * 128u + ((row & 7u) << 4);  // 16-B group gq of this row lives at chunk + (rowx ^ (gq << 4))
    const uint32_t sc_s = cblk_s + 4u * CL.scalars;
    uint4* scr = p.scratch + ((size_t)blockIdx.x * kGroups + tg) * (kTileRows * 32) + row;  // [32 uint4][128 rows]
    uint4* scr_t = scr + kTileRows * 32;                                                  // SPLIT: tails (group 1's scratch)
    // ---- training tape (SAVE): this row's slice of the current tile's chunk images / sign words
    const TapeLayout& TL = p.tape;
    uint8_t* tape_tile = nullptr;   // first chunk of the tile
    uint32_t* mask_row = nullptr;   // sign words of this row in slot 0; slot s is kTileRows * kMaskWords words further ([slot][row][word]:
                                    // the lanes of a warp write / read consecutive 32-B groups)
    // 32 columns (16 packed registers) starting at column col0 of the operand whose first chunk is `chunk`
    auto tape_st32 = [&](int chunk, int col0, const uint32_t (&o)[16]) {
      if constexpr (SAVE) {
        if (tape_tile != nullptr && chunk >= 0) {
          chunk_st32(tape_tile + tape_row_off(TL.n_a, chunk + (col0 >> 6), row), row, (uint32_t)(col0 & 63) >> 3, o);
        }
      }
    };
    auto mask_st = [&](int slot, int word, uint32_t bits) {
      if constexpr (SAVE) {
        if (mask_row != nullptr && slot >= 0) mask_row[(size_t)slot * (kTileRows * kMaskWords) + word] = bits;
      }
    };

    // the prologue kernel (previous launch in the stream) wrote the workspace: wait for that grid to finish
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // stage the constant block once
    {
      const float4* src = reinterpret_cast<const float4*>(p.workspace);
      float4* dst = reinterpret_cast<float4*>(cblk);
      for (int i = threadIdx.x; i < CL.n_floats / 4; i += kComputeThreads) dst[i] = __ldg(src + i);
    }
    named_bar_sync(3, kComputeThreads);

    auto warp_arrive = [&](uint64_t* bar) {
      __syncwarp();
      if (lane == 0) mbar_arrive(bar);
    };
    auto arrive_all = [&]() {
      fence_proxy_async_smem();
      tc_fence_before_sync();
      warp_arrive(&c2m_g[BAR_ALL]);
    };
    auto wait_all = [&]() {
      mbar_wait(&m2c_g[BAR_ALL], all_phase);
      all_phase ^= 1;
      tc_fence_after_sync();
    };
    auto gemm = [&]() { arrive_all(); wait_all(); };
    auto wait_half = [&](int nh) {
      mbar_wait(&m2c_g[BAR_H0 + nh], (half_phase >> nh) & 1u);
      half_phase ^= 1u << nh;
      tc_fence_after_sync();
    };
    auto bias_s = [&](int layer) -> uint32_t { return (P.bias[layer].frame ? fblk_s : cblk_s) + 4u * P.bias[layer].off; };
    // (a, b) -> packed 16-bit heads and, in SPLIT mode, the packed tails a - head(a), b - head(b)
    auto pack_ht = [&](float a, float b, uint32_t& hd, uint32_t& tl) {
      hd = Op::pack2(a, b);
      if constexpr (SPLIT) {
        const float2 f = Op::unpack2(hd);
        tl = Op::pack2(a - f.x, b - f.y);
      }
    };
    // 32 accumulator columns + bias -> relu -> 16 packed columns (+ 16 packed tails)
    // sign bits of 32 pre-activations: column pair i (columns 2i, 2i+1) -> bits 15-i and 31-i (1 = not positive)
    uint32_t sg_lo = 0u, sg_hi = 0u;
    auto sign2 = [&](float even, float odd) {
      if constexpr (SAVE) {
        sg_lo = __funnelshift_l(__float_as_uint(even), sg_lo, 1);
        sg_hi = __funnelshift_l(__float_as_uint(odd), sg_hi, 1);
      }
    };
    auto sign_word = [&]() { const uint32_t w = (sg_hi << 16) | (sg_lo & 0xFFFFu); sg_lo = 0u; sg_hi = 0u; return w; };
    auto relu_pack32 = [&](const uint32_t (&ra)[32], uint32_t bias, uint32_t (&o)[16], uint32_t (&ot)[16]) {
#pragma unroll
      for (int g4 = 0; g4 < 8; ++g4) {
        const float4 b = lds128(bias + 16u * g4);
        // packed fp32 adds (FADD2): two columns per instruction
        const float2 s0 = __fadd2_rn(make_float2(__uint_as_float(ra[4 * g4 + 0]), __uint_as_float(ra[4 * g4 + 1])), make_float2(b.x, b.y));
        const float2 s1 = __fadd2_rn(make_float2(__uint_as_float(ra[4 * g4 + 2]), __uint_as_float(ra[4 * g4 + 3])), make_float2(b.z, b.w));
        sign2(s0.x, s0.y);
        sign2(s1.x, s1.y);
        if constexpr (SPLIT) {
          pack_ht(fmaxf(s0.x, 0.f), fmaxf(s0.y, 0.f), o[2 * g4], ot[2 * g4]);
          pack_ht(fmaxf(s1.x, 0.f), fmaxf(s1.y, 0.f), o[2 * g4 + 1], ot[2 * g4 + 1]);
        } else {
          o[2 * g4] = Op::pack2_relu(s0.x, s0.y);
          o[2 * g4 + 1] = Op::pack2_relu(s1.x, s1.y);
        }
      }
    };
    // finished GEMM of n (<= 128) columns: relu(acc + bias) -> activations [0, n)
    auto epi_relu_act = [&](uint32_t bias, int n, int save_chunk, int mask_slot) {
      const int nb = n >> 5;
#pragma unroll 1
      for (int blk = SPLIT ? (g * nb) >> 1 : 0; blk < (SPLIT ? ((g + 1) * nb) >> 1 : nb); ++blk) {
        uint32_t ra[32], o[16], ot[SPLIT ? 16 : 1];
        tmem_ld32_issue(tD + 32 * blk, ra);
        tmem_ld_wait32(ra);
        if constexpr (SPLIT) {
          relu_pack32(ra, bias + 128u * blk, o, ot);
          tmem_st16(tA + kTail + 16 * blk, ot);
        } else {
          relu_pack32(ra, bias + 128u * blk, o, o);
        }
        tmem_st16(tA + 16 * blk, o);
        tape_st32(save_chunk, 32 * blk, o);
        mask_st(mask_slot, blk, sign_word());
      }
      tmem_st_wait();
    };
    // One 2*hn-wide layer issued as two N-halves on this group's accumulator (program.h pipe5).
    //   MODE 0: relu(acc + bias) -> activations (in place: half 0 is held in registers until the layer's MMAs are done)
    //   MODE 1: basefield.linear_final: relu features -> packed into the per-row scratch, fp32 dot with sdf.weight
    //   MODE 2: colorfield.linear_final: relu(acc + bias) + base features (scratch) -> activations (input of rgb.0)
    float sdf_acc = 0.f;
    auto chain_layer = [&](auto mode_tag, uint32_t bias, int save_chunk, int mask_slot) {
      constexpr int MODE = decltype(mode_tag)::value;
      auto math = [&](const uint32_t (&ra)[32], int col0, uint32_t (&o)[16], uint32_t (&ot)[16]) {  // col0: first feature of these 32 columns
        const uint32_t ba = bias + 4u * (uint32_t)col0;
        if (MODE == 0) {
          relu_pack32(ra, ba, o, ot);
        } else if (MODE == 1) {
          const uint32_t wa = cblk_s + 4u * (CL.sdf_w + col0);
          float s0 = 0.f, s1 = 0.f;
#pragma unroll
          for (int g4 = 0; g4 < 8; ++g4) {
            const float4 b = lds128(ba + 16u * g4), w = lds128(wa + 16u * g4);
            const float z0 = __uint_as_float(ra[4 * g4 + 0]) + b.x, z1 = __uint_as_float(ra[4 * g4 + 1]) + b.y;
            const float z2 = __uint_as_float(ra[4 * g4 + 2]) + b.z, z3 = __uint_as_float(ra[4 * g4 + 3]) + b.w;
            sign2(z0, z1);
            sign2(z2, z3);
            const float y0 = fmaxf(z0, 0.f), y1 = fmaxf(z1, 0.f), y2 = fmaxf(z2, 0.f), y3 = fmaxf(z3, 0.f);
            s0 += y0 * w.x + y2 * w.z;
            s1 += y1 * w.y + y3 * w.w;
            pack_ht(y0, y1, o[2 * g4], ot[2 * g4]);
            pack_ht(y2, y3, o[2 * g4 + 1], ot[2 * g4 + 1]);
          }
          if constexpr (SPLIT) sts32(sdf_part_s + 4u * ((uint32_t)(col0 >> 5) * kTileRows + row), s0 + s1);  // summed in block order
          else sdf_acc += s0 + s1;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            scr[(size_t)((col0 >> 3) + j) * kTileRows] = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
            if constexpr (SPLIT) scr_t[(size_t)((col0 >> 3) + j) * kTileRows] = make_uint4(ot[4 * j], ot[4 * j + 1], ot[4 * j + 2], ot[4 * j + 3]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint4 bf = scr[(size_t)((col0 >> 3) + j) * kTileRows];
            uint4 bt = make_uint4(0u, 0u, 0u, 0u);
            if constexpr (SPLIT) bt = scr_t[(size_t)((col0 >> 3) + j) * kTileRows];
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const int g4 = 2 * j + hh;
              const float4 b = lds128(ba + 16u * g4);
              float2 f0 = Op::unpack2(hh ? bf.z : bf.x), f1 = Op::unpack2(hh ? bf.w : bf.y);
              if constexpr (SPLIT) {
                const float2 t0 = Op::unpack2(hh ? bt.z : bt.x), t1 = Op::unpack2(hh ? bt.w : bt.y);
                f0.x += t0.x; f0.y += t0.y; f1.x += t1.x; f1.y += t1.y;
              }
              const float z0 = __uint_as_float(ra[4 * g4 + 0]) + b.x, z1 = __uint_as_float(ra[4 * g4 + 1]) + b.y;
              const float z2 = __uint_as_float(ra[4 * g4 + 2]) + b.z, z3 = __uint_as_float(ra[4 * g4 + 3]) + b.w;
              sign2(z0, z1);
              sign2(z2, z3);
              pack_ht(fmaxf(z0, 0.f) + f0.x, fmaxf(z1, 0.f) + f0.y, o[2 * g4], ot[2 * g4]);
              pack_ht(fmaxf(z2, 0.f) + f1.x, fmaxf(z3, 0.f) + f1.y, o[2 * g4 + 1], ot[2 * g4 + 1]);
            }
          }
        }
      };
      if constexpr (SPLIT) {
        // Group g takes the BPG blocks [g * BPG, (g + 1) * BPG) of each N-half.  Half 1 accumulates in columns [128, 256),
        // so its MMAs run while half 0 is drained; half 0's heads and tails wait in registers until the layer's MMAs have
        // read its input.
        constexpr int BPG = NBLK / 2;
        const int blk0 = g * BPG;
        uint32_t hd[BPG][16], tl[BPG][16];
        uint32_t mw[SAVE ? 2 * BPG : 1];
        wait_half(0);
#pragma unroll
        for (int i = 0; i < BPG; ++i) {  // one block per TMEM round trip: keeps half 0's heads and tails in registers without spills
          uint32_t ra[32];
          tmem_ld32_issue(tD + 32 * (blk0 + i), ra);
          tmem_ld_wait32(ra);
          math(ra, 32 * (blk0 + i), hd[i], tl[i]);
          tape_st32(save_chunk, 32 * (blk0 + i), hd[i]);
          if constexpr (SAVE) mw[i] = sign_word();
        }
        // ---- N-half 1: the layer's input has been read, activations can be overwritten
        wait_half(1);
        if (MODE != 1) {
#pragma unroll
          for (int i = 0; i < BPG; ++i) {
            tmem_st16(tA + 16 * (blk0 + i), hd[i]);
            tmem_st16(tA + kTail + 16 * (blk0 + i), tl[i]);
          }
        }
#pragma unroll
        for (int i = 0; i < BPG; ++i) {  // one block per round trip too: the other group's warp covers the latency
          const int blk = blk0 + i;
          uint32_t ra[32], o[16], ot[16];
          tmem_ld32_issue(tD + kTmemGroup + 32 * blk, ra);
          tmem_ld_wait32(ra);
          math(ra, HN + 32 * blk, o, ot);
          if (MODE != 1) {
            tmem_st16(tA + (HN >> 1) + 16 * blk, o);
            tmem_st16(tA + kTail + (HN >> 1) + 16 * blk, ot);
          }
          tape_st32(save_chunk, HN + 32 * blk, o);
          if constexpr (SAVE) mw[BPG + i] = sign_word();
        }
        if constexpr (SAVE) {  // this group's sign words of each half: words [blk0, blk0 + BPG) and NBLK further
          if (mask_row != nullptr && mask_slot >= 0) {
            uint32_t* mp = mask_row + (size_t)mask_slot * (kTileRows * kMaskWords);
            if constexpr (BPG == 2) {
              *reinterpret_cast<uint2*>(mp + blk0) = make_uint2(mw[0], mw[1]);
              *reinterpret_cast<uint2*>(mp + NBLK + blk0) = make_uint2(mw[2], mw[3]);
            } else {
#pragma unroll
              for (int i = 0; i < BPG; ++i) { mp[blk0 + i] = mw[i]; mp[NBLK + blk0 + i] = mw[BPG + i]; }
            }
          }
        }
        if (MODE != 1) tmem_st_wait();
        tc_fence_before_sync();
        warp_arrive(&c2m_g[BAR_H1]);
      } else {
        // ---- N-half 0: drain the accumulator so the MMAs of half 1 can start
        uint32_t hold[NBLK][16];
        uint32_t mwords[SAVE ? 2 * NBLK : 1];
        wait_half(0);
#pragma unroll
        for (int bp = 0; bp < NBLK; bp += 2) {  // two 32-column blocks per TMEM round trip
          uint32_t rp[2][32];
          tmem_ld32_issue(tD + 32 * bp, rp[0]);
          tmem_ld32_issue(tD + 32 * (bp + 1), rp[1]);
          tmem_ld_wait32(rp[0]);
          tmem_ld_wait32(rp[1]);
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            const int blk = bp + h2;
            math(rp[h2], 32 * blk, hold[blk], hold[blk]);
            tape_st32(save_chunk, 32 * blk, hold[blk]);
            if constexpr (SAVE) mwords[blk] = sign_word();
          }
        }
        tc_fence_before_sync();
        warp_arrive(&c2m_g[BAR_H0]);
        // ---- N-half 1: the layer's input has been read, activations can be overwritten
        wait_half(1);
        if (MODE != 1) {
#pragma unroll
          for (int blk = 0; blk < NBLK; ++blk) tmem_st16(tA + 16 * blk, hold[blk]);
        }
#pragma unroll
        for (int bp = 0; bp < NBLK; bp += 2) {
          uint32_t rp[2][32];
          tmem_ld32_issue(tD + 32 * bp, rp[0]);
          tmem_ld32_issue(tD + 32 * (bp + 1), rp[1]);
          tmem_ld_wait32(rp[0]);
          tmem_ld_wait32(rp[1]);
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            const int blk = bp + h2;
            uint32_t o[16];
            math(rp[h2], HN + 32 * blk, o, o);
            if (MODE != 1) tmem_st16(tA + (HN >> 1) + 16 * blk, o);
            tape_st32(save_chunk, HN + 32 * blk, o);
            if constexpr (SAVE) mwords[NBLK + blk] = sign_word();
          }
        }
        if constexpr (SAVE) {  // the layer's sign words in one (or two) 16-B stores
          if (mask_row != nullptr && mask_slot >= 0) {
            uint4* mp = reinterpret_cast<uint4*>(mask_row + (size_t)mask_slot * (kTileRows * kMaskWords));
            mp[0] = make_uint4(mwords[0], mwords[1], mwords[2], mwords[3]);
            if (NBLK > 2) mp[1] = make_uint4(mwords[4 % (2 * NBLK)], mwords[5 % (2 * NBLK)], mwords[6 % (2 * NBLK)], mwords[7 % (2 * NBLK)]);
          }
        }
        if (MODE != 1) tmem_st_wait();
        tc_fence_before_sync();
        warp_arrive(&c2m_g[BAR_H1]);
      }
    };

    // 16-bit element `c` (0..63) of this row in an operand chunk
    auto put16 = [&](uint32_t chunk_s, int c, float val) {
      const uint32_t a = chunk_s + (rowx ^ ((uint32_t)(c >> 3) << 4)) + 2u * (c & 7);
      const uint16_t hd = Op::cvt(val);
      sts16(a, hd);
      if constexpr (SPLIT) sts16(a + kArenaGroup, Op::cvt(val - Op::f32(hd)));  // tail chunk: group 1's arena
    };
    // Fourier features of x: column e < 3 -> x_e, else frequency (e-3)/6, sin for (e-3)%6 < 3 (PosEmbedding.forward,
    // nnutils/embedding.py:69-125).  Columns 0..62 live in CH_PE, 63.. in CH_EXTRA.
    auto embed = [&](const float3& x, int nfreq) {
      auto put = [&](int e, float val) { put16(e < 63 ? pe_s : extra_s, e < 63 ? e : e - 63, val); };
      put(0, x.x); put(1, x.y); put(2, x.z);
      // sin/cos of 2^k x: evaluated directly for every fourth frequency, the three in between follow from the
      // double-angle identities (error doubles per step: <= 8 ulp-level errors of the direct value, far below the
      // 16-bit operand rounding of 2^-11)
      float fr = 1.0f;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, c0 = 1.f, c1 = 1.f, c2 = 1.f;
#pragma unroll 1
      for (int kf = 0; kf < nfreq; ++kf) {
        if ((kf & 3) == 0) {
          sincosf(fr * x.x, &s0, &c0);
          sincosf(fr * x.y, &s1, &c1);
          sincosf(fr * x.z, &s2, &c2);
        } else {
          const float t0 = 2.f * s0 * c0, t1 = 2.f * s1 * c1, t2 = 2.f * s2 * c2;
          c0 = 1.f - 2.f * s0 * s0; c1 = 1.f - 2.f * s1 * s1; c2 = 1.f - 2.f * s2 * s2;
          s0 = t0; s1 = t1; s2 = t2;
        }
        const int e0 = 3 + 6 * kf;
        put(e0, s0); put(e0 + 1, s1); put(e0 + 2, s2);
        put(e0 + 3, c0); put(e0 + 4, c1); put(e0 + 5, c2);
        fr *= 2.0f;
      }
    };
    // DenseWarp.forward (nnutils/warping.py:143-170): x + 0.1 * CondMLP([PE6(x), t, inst]); the per-frame codes are
    // folded into the linear_1 bias row `bias1`; lid0 = canonical id of the map's linear_1.
    // copy this row's 128 B (8 swizzled 16-B groups, `ngroups` of them in use) of an embedding chunk to the tape
    auto tape_copy_row = [&](int chunk, uint32_t chunk_s, int ngroups) {
      if constexpr (SAVE) {
        if (tape_tile != nullptr && chunk >= 0) {
          uint8_t* rp = tape_tile + tape_row_off(TL.n_a, chunk, row);
          for (int gq = 0; gq < ngroups; ++gq) {
            const uint32_t slot = ((uint32_t)gq ^ (row & 7u)) << 4;
            *reinterpret_cast<uint4*>(rp + slot) = lds128u(chunk_s + row * 128u + slot);
          }
        }
      }
    };
    auto dense_warp = [&](const float3& x, uint32_t bias1, int lid0, int w) -> float3 {
      if (lead) {
        embed(x, 6);
        put16(pe_s, 39, 0.f);  // 39 embedding columns; the third k-step reads up to column 47
        sts128(pe_s + (rowx ^ (5u << 4)), make_uint4(0u, 0u, 0u, 0u));
        if constexpr (SPLIT) sts128(pe_s + kArenaGroup + (rowx ^ (5u << 4)), make_uint4(0u, 0u, 0u, 0u));
        tape_copy_row(TL.a_dpe[w], pe_s, 6);
      }
      arrive_all();
#pragma unroll 1
      for (int l = 0; l < 2; ++l)
        chain_layer(IC<0>{}, l == 0 ? bias1 : bias_s(lid0 + 1), l == 0 ? TL.a_dh1[w] : TL.a_dh2[w], l == 0 ? TL.m_dh1[w] : TL.m_dh2[w]);
      wait_all();
      if (!lead) return x;
      float m[16];
      tmem_ld16(tD, m);
      const uint32_t b3 = bias_s(lid0 + 2);
      return make_float3(x.x + 0.1f * (m[0] + lds32(b3)), x.y + 0.1f * (m[1] + lds32(b3 + 4)), x.z + 0.1f * (m[2] + lds32(b3 + 8)));
    };

    for (int it = 0; it < iters; ++it) {
      const int tile_raw = (kActive * it + tg) * (int)gridDim.x + (int)blockIdx.x;
      const bool dead_tile = tile_raw >= p.n_tiles;
      const int tile = dead_tile ? p.n_tiles - 1 : tile_raw;
      const int f = tile / p.tiles_per_frame;
      const int r_raw = (tile - f * p.tiles_per_frame) * kTileRows + (int)row;
      const bool live = lead && !dead_tile && r_raw < p.ND;  // this thread writes the row's per-sample outputs
      const int r_in = r_raw < p.ND ? r_raw : p.ND - 1;
      const int n = r_in / p.rays.D;
      const int k = r_in - n * p.rays.D;
      const size_t s = (size_t)f * p.ND + r_in;
      if constexpr (SAVE) {
        tape_tile = dead_tile ? nullptr : p.tape_a + (size_t)tile * TL.n_a * kChunkBytes;
        mask_row = dead_tile ? nullptr : p.tape_mask + ((size_t)tile * TL.n_mask * kTileRows + row) * kMaskWords;
      }

      // ------------------------------------------------ stage this frame's block in shared memory
      named_bar_sync(1 + tg, kTileThreads);  // the tile's warps are done with the previous block
      {
        const float4* src = reinterpret_cast<const float4*>(p.workspace + CL.n_floats + (size_t)f * FL.n_floats);
        float4* dst = reinterpret_cast<float4*>(fblk_g);
        for (int i = ttid; i < FL.n_floats / 4; i += kTileThreads) dst[i] = __ldg(src + i);
      }
      named_bar_sync(1 + tg, kTileThreads);

      // ------------------------------------------------ sample placement (sample_cam_rays)
      const bool pts = p.points != nullptr;  // b200r_points_fwd: canonical points are given, only NeRF.forward runs
      float h0 = 0.f, h1 = 0.f, depth = 0.f, delta = 0.f;
      float3 xyz_cam = make_float3(0.f, 0.f, 0.f), xyz_t = xyz_cam, dir_f = xyz_cam;
      if (lead && !pts) {
        const float* hx = p.rays.hxy + ((size_t)f * p.rays.N + n) * 3;
        h0 = __ldg(hx); h1 = __ldg(hx + 1);
        const float h2 = __ldg(hx + 2);
        const float* cam = fblk_g + FL.cam;
        float3 d = make_float3(h0 * cam[0] + h1 * cam[1] + h2 * cam[2], h0 * cam[3] + h1 * cam[4] + h2 * cam[5],
                               h0 * cam[6] + h1 * cam[7] + h2 * cam[8]);
        const float dn = sqrtf(d.x * d.x + d.y * d.y + d.z * d.z);
        const float nearv = cam[9], farv = cam[10];
        const int Dn = p.rays.D;
        const float step = 1.0f / (float)(Dn - 1);
        auto lin = [&](int i) { return i < Dn / 2 ? step * (float)i : 1.0f - step * (float)(Dn - 1 - i); };
        auto depth_at = [&](int i) { float z = lin(i); return nearv * (1.0f - z) + farv * z; };
        if (p.rays.depth) {  // given sample depths (importance sampling): sample_cam_rays(depth=...)
          const float* dp = p.rays.depth + ((size_t)f * p.rays.N + n) * Dn;
          depth = __ldg(dp + k);
          delta = (k + 1 < Dn ? __ldg(dp + k + 1) - depth : depth - __ldg(dp + k - 1)) * dn;
        } else {
          depth = depth_at(k);
          delta = (k + 1 < Dn ? depth_at(k + 1) - depth : depth - depth_at(k - 1)) * dn;
        }
        xyz_cam = make_float3(d.x * depth, d.y * depth, d.z * depth);
        const float3 dir_cam = make_float3(d.x / dn, d.y / dn, d.z / dn);

        // ---------------------------------------------- camera -> field (cam_to_field)
        const Q4 qc = {cam[11], cam[12], cam[13], cam[14]};
        const Q4 qi = qconj(qc);
        const float3 ti = qrot(qi, make_float3(-cam[15], -cam[16], -cam[17]));
        xyz_t = qrot(qi, xyz_cam);
        xyz_t.x += ti.x; xyz_t.y += ti.y; xyz_t.z += ti.z;
        dir_f = qrot(qi, dir_cam);
      } else if (lead) {
        const float* px = p.points + s * 3;
        xyz_t = make_float3(__ldg(px), __ldg(px + 1), __ldg(px + 2));
        if (p.point_dirs) {
          const float* pd = p.point_dirs + s * 3;
          dir_f = make_float3(__ldg(pd), __ldg(pd + 1), __ldg(pd + 2));
        }
      }

      // ------------------------------------------------ skinning warps (SkinningWarp.forward), three per sample:
      //   w = 0 backward warp (time-t -> canonical), w = 1 forward warp with the pair partner's articulation (flow),
      //   w = 2 forward warp with the frame's own articulation (cycle).
      // bone coordinates -> delta MLP on the tensor pipe -> softmax -> dual-quaternion blend.
      constexpr int NP = B > 0 ? (3 * B + 15) / 16 * 8 : 1;  // packed pairs of the zero-padded bone-coordinate row
      auto skin_warp = [&](const float3& x, uint32_t binv, uint32_t se3, uint32_t bias1, float& entropy, float& delta_skin, int w) -> float3 {
        float dist2[B > 0 ? B : 1];
        if (lead) {
          uint32_t u[NP], ut[SPLIT ? NP : 1];
#pragma unroll
          for (int i = 0; i < NP; ++i) u[i] = 0u;
          if constexpr (SPLIT) {
#pragma unroll
            for (int i = 0; i < NP; ++i) ut[i] = 0u;
          }
#pragma unroll
          for (int b2 = 0; b2 < (B + 1) / 2; ++b2) {
            float v[6];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const int b = 2 * b2 + j;
              if (b < B) {
                const uint32_t ba = binv + 48u * b;
                const float4 r0 = lds128(ba), r1 = lds128(ba + 16), r2 = lds128(ba + 32);
                v[3 * j + 0] = r0.x * x.x + r0.y * x.y + r0.z * x.z + r0.w;
                v[3 * j + 1] = r1.x * x.x + r1.y * x.y + r1.z * x.z + r1.w;
                v[3 * j + 2] = r2.x * x.x + r2.y * x.y + r2.z * x.z + r2.w;
                dist2[b] = v[3 * j] * v[3 * j] + v[3 * j + 1] * v[3 * j + 1] + v[3 * j + 2] * v[3 * j + 2];
              } else {
                v[3 * j] = v[3 * j + 1] = v[3 * j + 2] = 0.f;
              }
            }
            pack_ht(v[0], v[1], u[3 * b2], ut[SPLIT ? 3 * b2 : 0]);
            pack_ht(v[2], v[3], u[3 * b2 + 1], ut[SPLIT ? 3 * b2 + 1 : 0]);
            pack_ht(v[4], v[5], u[3 * b2 + 2], ut[SPLIT ? 3 * b2 + 2 : 0]);
          }
          tmem_st32(tA, u);
          if (NP > 32) tmem_st8(tA + 32, u + (NP > 32 ? 32 : 0));
          if constexpr (SPLIT) {
            tmem_st32(tA + kTail, ut);
            if (NP > 32) tmem_st8(tA + kTail + 32, ut + (NP > 32 ? 32 : 0));
          }
          if constexpr (SAVE) {  // bone coordinates: the delta MLP's input operand (zero padded)
            if (tape_tile != nullptr) {
#pragma unroll
              for (int j = 0; j < NP / 4; ++j) {
                uint8_t* rp = tape_tile + tape_row_off(TL.n_a, TL.a_xb[w] + (j >> 3), row);
                *reinterpret_cast<uint4*>(rp + ((((uint32_t)j & 7u) ^ (row & 7u)) << 4)) = make_uint4(u[4 * j], u[4 * j + 1], u[4 * j + 2], u[4 * j + 3]);
              }
            }
          }
          tmem_st_wait();
        }
        // delta_field.linear_1 / linear_2 (ReLU) and linear_final
        gemm();
        epi_relu_act(bias1, 64, TL.a_h1[w], TL.m_h1[w]);
        gemm();
        epi_relu_act(bias_s(lid_delta + 1), 64, TL.a_h2[w], TL.m_h2[w]);
        gemm();
        if (!lead) return x;
        float dl[32];
        tmem_ld32(tD, dl);
        const uint32_t b3 = bias_s(lid_delta + 2);
        float mx = -INFINITY, dsum = 0.f;
        int amax = 0;
        if constexpr (SAVE) {  // raw delta-MLP outputs (pre-ReLU), 16-bit: the backward recomputes the blend from them
          uint32_t zz[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float a0 = 2 * j < B ? dl[2 * j] + lds32(b3 + 8u * j) : 0.f, a1 = 2 * j + 1 < B ? dl[2 * j + 1] + lds32(b3 + 8u * j + 4u) : 0.f;
            zz[j] = Op::pack2(a0, a1);
          }
          tape_st32(TL.a_z[w], 0, zz);
        }
#pragma unroll
        for (int j = 0; j < B; ++j) {
          const float dv = 0.1f * fmaxf(dl[j] + lds32(b3 + 4u * j), 0.f);
          dsum += dv * dv;
          const float lg = -(dist2[j] + dv);
          dist2[j] = lg;
          if (lg > mx) { mx = lg; amax = j; }  // first maximum wins, like argmax
        }
        const float4 qa = lds128(se3 + 32u * amax);
        float se = 0.f;
        float4 qr = make_float4(0.f, 0.f, 0.f, 0.f), qd = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < B; ++j) {
          const uint32_t sa = se3 + 32u * j;
          const float e = __expf(dist2[j] - mx);
          se += e;
          const float4 r = lds128(sa), dq = lds128(sa + 16);
          const float dot = qa.x * r.x + qa.y * r.y + qa.z * r.z + qa.w * r.w;
          const float wgt = dot > 0.f ? e : -e;  // the softmax denominator cancels in the normalisation below
          qr.x += wgt * r.x; qr.y += wgt * r.y; qr.z += wgt * r.z; qr.w += wgt * r.w;
          qd.x += wgt * dq.x; qd.y += wgt * dq.y; qd.z += wgt * dq.z; qd.w += wgt * dq.w;
        }
        entropy = __logf(se);  // logsumexp - max  (cross_entropy_skin_loss)
        delta_skin = dsum / (float)(B > 0 ? B : 1);
        // stored order is (w,x,y,z) in (.x,.y,.z,.w)
        const float inv = rsqrtf(qr.x * qr.x + qr.y * qr.y + qr.z * qr.z + qr.w * qr.w);
        const Q4 Qr = {qr.x * inv, qr.y * inv, qr.z * inv, qr.w * inv};
        const Q4 Qd = {qd.x * inv, qd.y * inv, qd.z * inv, qd.w * inv};
        const Q4 tq = qmul(Qd, qconj(Qr));
        float3 o = qrot(Qr, x);
        o.x += 2.f * tq.x; o.y += 2.f * tq.y; o.z += 2.f * tq.z;
        return o;
      };

      float3 xyz = xyz_t, x_next = xyz_t;
      float ent_b = 0.f, dsk_b = 0.f, ent_out = 0.f, dsk_out = 0.f, cyc = 0.f;
      const int wm = p.warp_mode;  // b200r_warp_fwd: one warp of the given points, nothing else
      if (pts && !wm) {
        // canonical points are given
      } else if constexpr (B > 0) {
        // ComposedWarp (warping.py:445-483) interleaves the DenseWarp soft deformation: backward = skin then dense,
        // forward = dense then skin.  One loop over stages keeps a single inlined copy of either body.
        constexpr int NST = DENSE ? 6 : 3;
        constexpr int PER = DENSE ? 2 : 1;  // stages per warp
        const int stg_lo = wm == MODE_WARP_FWD ? 2 * PER : 0, stg_hi = wm == MODE_WARP_BWD ? PER : NST;
        float3 cur = xyz_t;
#pragma unroll 1
        for (int stg = stg_lo; stg < stg_hi; ++stg) {
          const int w = DENSE ? (stg >> 1) : stg;
          if (DENSE && (stg == 1 || stg == 2 || stg == 4)) {
            const uint32_t bias1 = stg == 1 ? bias_s(lid_dense + 3) : (stg == 2 ? fblk_s + 4u * FL.dense1_partner : bias_s(lid_dense));
            cur = dense_warp(stg == 1 ? cur : xyz, bias1, stg == 1 ? lid_dense + 3 : lid_dense, w);
            if (stg == 1) xyz = cur;
            continue;
          }
          const float3 src = w == 0 ? xyz_t : (DENSE ? cur : xyz);
          const uint32_t binv = fblk_s + 4u * (w == 0 ? FL.binv_t : (w == 1 ? FL.binv_rest_partner : FL.binv_rest));
          const uint32_t se3 = fblk_s + 4u * (w == 0 ? FL.se3_bwd : (w == 1 ? FL.se3_fwd_partner : FL.se3_fwd));
          const uint32_t bias1 = w == 0 ? bias_s(lid_delta) : fblk_s + 4u * FL.delta1_fwd;  // forward warps: mean time code
          float e, dk;
          const float3 o = skin_warp(src, binv, se3, bias1, e, dk, w);
          if (SAVE && DENSE && live && p.out.warp_pts) {  // inputs of the dense maps / forward skinning warps (the backward recomputes from them)
            float* wp = p.out.warp_pts + s * 9 + 3 * w;  // w = 0: skinned point before the soft deformation; 1, 2: deformed points
            const float3 sv = w == 0 ? o : src;
            wp[0] = sv.x; wp[1] = sv.y; wp[2] = sv.z;
          }
          if (w == 0) { cur = o; xyz = o; ent_b = e; dsk_b = dk; }
          else if (w == 1) { x_next = o; }
          else {
            const float dx = o.x - xyz_t.x, dy = o.y - xyz_t.y, dz = o.z - xyz_t.z;
            cyc = sqrtf(dx * dx + dy * dy + dz * dz);
            ent_out = 0.5f * (e + ent_b);
            dsk_out = 0.5f * (dk + dsk_b);
            if (wm) { xyz = o; ent_b = e; dsk_b = dk; }  // warp entry, forward: the warped point and its own aux
          }
        }
      } else {
        x_next = xyz;
      }
      if (wm) {  // b200r_warp_fwd: warped point + the call's aux values, then on to the next tile
        if (live) {
          if (p.out.xyz) { p.out.xyz[s * 3] = xyz.x; p.out.xyz[s * 3 + 1] = xyz.y; p.out.xyz[s * 3 + 2] = xyz.z; }
          if (p.out.skin_entropy) p.out.skin_entropy[s] = ent_b;
          if (p.out.delta_skin) p.out.delta_skin[s] = dsk_b;
        }
        continue;
      }

      // ------------------------------------------------ outputs that are final before the MLPs run
      auto st3 = [&](float* dst, float a, float b, float c) { if (dst && live) { dst[s * 3] = a; dst[s * 3 + 1] = b; dst[s * 3 + 2] = c; } };
      auto st1 = [&](float* dst, float a) { if (dst && live) dst[s] = a; };
      if (lead && pts) {
        st3(p.out.xyz, xyz.x, xyz.y, xyz.z);
      } else if (lead) {
        // field_to_cam with the partner frame's camera, pinhole projection, flow (nerf.py:948-997)
        const float* cn = fblk_g + FL.cam_partner;
        const Q4 qn = {cn[11], cn[12], cn[13], cn[14]};
        float3 xc = qrot(qn, x_next);
        xc.x += cn[15]; xc.y += cn[16]; xc.z += cn[17];
        const float k0 = cn[0], k1 = cn[4], k2 = cn[2], k3 = cn[5];
        const float fx = 1.0f / k0, fy = 1.0f / k1, cx = -k2 / k0, cy = -k3 / k1;
        const float hxn = (fx * xc.x + cx * xc.z) / (xc.z + 1e-6f);
        const float hyn = (fy * xc.y + cy * xc.z) / (xc.z + 1e-6f);
        const float fl0 = hxn - h0, fl1 = hyn - h1;
        bool valid = xc.z > 1e-6f;
        if (p.rays.flow_thresh >= 0.f) valid = valid && (sqrtf(fl0 * fl0 + fl1 * fl1) < p.rays.flow_thresh);
        st3(p.out.flow, fl0, fl1, valid ? 1.f : 0.f);
        // Gaussian bone density (compute_gauss_density): max_b exp(-d2_b / 2) = exp(-min_b d2_b / 2)
        if constexpr (B > 0) {
          float best = INFINITY;
          const uint32_t ctr = cblk_s + 4u * CL.center;
#pragma unroll 5
          for (int b = 0; b < B; ++b) {
            const float4 c = lds128(ctr + 16u * b);
            const float dx = xyz.x - c.x, dy = xyz.y - c.y, dz = xyz.z - c.z;
            best = fminf(best, dx * dx + dy * dy + dz * dz);
          }
          st1(p.out.gauss_density, expf(-0.5f * (best / (0.01f * 0.01f))) * lds32(sc_s + 4u * SC_WARP_IBETA));
        }
        st3(p.out.xyz, xyz.x, xyz.y, xyz.z);
        st3(p.out.xyz_cam, xyz_cam.x, xyz_cam.y, xyz_cam.z);
        st3(p.out.xyz_t, xyz_t.x, xyz_t.y, xyz_t.z);
        st3(p.out.dir, dir_f.x, dir_f.y, dir_f.z);
        st1(p.out.depth, depth * lds32(sc_s + 4u * SC_INV_SCALE));
        st1(p.out.deltas, delta);
        st1(p.out.cyc_dist, cyc);
        st1(p.out.delta_skin, dsk_out);
        st1(p.out.skin_entropy, ent_out);
      }

      // ------------------------------------------------ positional embedding of the canonical point
      if (lead) {
        embed(xyz, LMAX);
        sts16(pe_s + (rowx ^ (7u << 4)) + 14u, (uint16_t)0);  // zero pad column 63 of CH_PE
        if constexpr (SPLIT) sts16(pe_s + kArenaGroup + (rowx ^ (7u << 4)) + 14u, (uint16_t)0);
        if (LMAX > 10) {  // CH_EXTRA holds 12 values (columns 63..74); its k-step reads 16 columns
          sts32(extra_s + (rowx ^ (1u << 4)) + 8u, 0.f);
          sts32(extra_s + (rowx ^ (1u << 4)) + 12u, 0.f);
          if constexpr (SPLIT) {
            sts32(extra_s + kArenaGroup + (rowx ^ (1u << 4)) + 8u, 0.f);
            sts32(extra_s + kArenaGroup + (rowx ^ (1u << 4)) + 12u, 0.f);
          }
        }

        tape_copy_row(TL.a_pe, pe_s, 8);
        if (LMAX > 10) tape_copy_row(TL.a_extra, extra_s, 2);
      }
      // ------------------------------------------------ visibility MLP (VisField.forward)
      if (!pts) {
      gemm();
      epi_relu_act(bias_s(lid_vis), 64, TL.a_vis[0], TL.m_vis[0]);
      gemm();
      if (lead) {
        const uint32_t b2 = bias_s(lid_vis + 1), vw = cblk_s + 4u * CL.vis_w;
        float a0 = 0.f, a1 = 0.f;
#pragma unroll 1
        for (int c0 = 0; c0 < 64; c0 += 32) {
          float v[32];
          tmem_ld32(tD + c0, v);
          uint32_t hs[16];
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 ba = lds128(b2 + 4u * (c0 + j)), wa = lds128(vw + 4u * (c0 + j));
            const float z0 = v[j] + ba.x, z1 = v[j + 1] + ba.y, z2 = v[j + 2] + ba.z, z3 = v[j + 3] + ba.w;
            a0 += fmaxf(z0, 0.f) * wa.x + fmaxf(z2, 0.f) * wa.z;
            a1 += fmaxf(z1, 0.f) * wa.y + fmaxf(z3, 0.f) * wa.w;
            if constexpr (SAVE) {
              sign2(z0, z1);
              sign2(z2, z3);
              hs[j >> 1] = Op::pack2_relu(z0, z1);
              hs[(j >> 1) + 1] = Op::pack2_relu(z2, z3);
            }
          }
          if constexpr (SAVE) {
            tape_st32(TL.a_vis[1], c0, hs);
            mask_st(TL.m_vis[1], c0 >> 5, sign_word());
          }
        }
        st1(p.out.vis, a0 + a1 + lds32(sc_s + 4u * SC_VIS_B));
      }
      }

      // ------------------------------------------------ feature field (FeatureNeRF.compute_feat)
      if (p.desc.has_feature && !pts) {
#pragma unroll 1
        for (int i = 0; i < 5; ++i) {
          gemm();
          epi_relu_act(bias_s(lid_feat + i), 128, TL.a_feat[i], TL.m_feat[i]);
        }
        gemm();
        if (lead) {
          float v16[16];
          tmem_ld16(tD, v16);
          const uint32_t bf = bias_s(lid_feat + 5);
          float nn = 0.f;
#pragma unroll
          for (int j = 0; j < 16; ++j) { v16[j] += lds32(bf + 4u * j); nn += v16[j] * v16[j]; }
          const float inv = rsqrtf(nn);
          if (p.out.feat_norm && live) p.out.feat_norm[s] = inv;
          if (p.out.feature && live) {
            float4* fo = reinterpret_cast<float4*>(p.out.feature + s * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j) fo[j] = make_float4(v16[4 * j] * inv, v16[4 * j + 1] * inv, v16[4 * j + 2] * inv, v16[4 * j + 3] * inv);
          }
        }
      }

      // ------------------------------------------------ density + colour chains (NeRF.forward, nnutils/nerf.py:167-215)
      arrive_all();  // embedding operands written, accumulator and activations free
      sdf_acc = 0.f;
#pragma unroll 1
      for (int j = 0; j < p.desc.D; ++j) chain_layer(IC<0>{}, bias_s(lid_base + j), TL.a_base[j], TL.m_base[j]);
      chain_layer(IC<1>{}, bias_s(lid_base + p.desc.D), TL.a_base[p.desc.D], TL.m_base[p.desc.D]);
      if constexpr (SPLIT) {  // both groups' partial dot products, summed in block order (as the one-group order)
        if (lead) {
          named_bar_sync(4 + q, 64);  // warps q and 4 + q
#pragma unroll
          for (int blk = 0; blk < 2 * NBLK; ++blk) sdf_acc += lds32(sdf_part_s + 4u * ((uint32_t)blk * kTileRows + row));
        } else {
          named_bar_arrive(4 + q, 64);
        }
      }
      const float sdf = sdf_acc + lds32(sc_s + 4u * SC_SDF_B);
      const float ibeta = lds32(sc_s + 4u * SC_IBETA);
      const float sgn = sdf > 0.f ? 1.f : (sdf < 0.f ? -1.f : 0.f);
      st1(p.out.density, (0.5f + 0.5f * sgn * expm1f(-fabsf(sdf) * ibeta)) * ibeta);
      st1(p.out.sdf, sdf);
#pragma unroll 1
      for (int j = 0; j < 2; ++j) chain_layer(IC<0>{}, bias_s(lid_color + j), TL.a_col[j], TL.m_col[j]);
      chain_layer(IC<2>{}, bias_s(lid_color + 2), TL.a_f2, TL.m_col[2]);
      // rgb.0 on (base + colour features), then rgb.2 + sigmoid
      wait_all();
      if (lead) {
        const uint32_t b0 = bias_s(lid_rgb0), w2 = cblk_s + 4u * CL.rgb2_w, wd = cblk_s + 4u * CL.dir_w;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 1
        for (int c0 = 0; c0 < HN; c0 += 32) {
          float v[32];
          tmem_ld32(tD + c0, v);
          uint32_t hs0[16];
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 bv = lds128(b0 + 4u * (c0 + j));
            const float4 wr = lds128(w2 + 4u * (c0 + j)), wg = lds128(w2 + 4u * (HN + c0 + j)), wb = lds128(w2 + 4u * (2 * HN + c0 + j));
            float pre[4] = {v[j] + bv.x, v[j + 1] + bv.y, v[j + 2] + bv.z, v[j + 3] + bv.w};
            if (p.desc.L_dir == 0) {
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const uint32_t da = wd + 12u * (c0 + j + u);
                pre[u] += lds32(da) * dir_f.x + lds32(da + 4) * dir_f.y + lds32(da + 8) * dir_f.z;
              }
            }
            const float h0_ = fmaxf(pre[0], 0.f), h1_ = fmaxf(pre[1], 0.f), h2_ = fmaxf(pre[2], 0.f), h3_ = fmaxf(pre[3], 0.f);
            if constexpr (SAVE) {
              sign2(pre[0], pre[1]);
              sign2(pre[2], pre[3]);
              hs0[j >> 1] = Op::pack2(h0_, h1_);
              hs0[(j >> 1) + 1] = Op::pack2(h2_, h3_);
            }
            a0 += h0_ * wr.x + h1_ * wr.y + h2_ * wr.z + h3_ * wr.w;
            a1 += h0_ * wg.x + h1_ * wg.y + h2_ * wg.z + h3_ * wg.w;
            a2 += h0_ * wb.x + h1_ * wb.y + h2_ * wb.z + h3_ * wb.w;
          }
          if constexpr (SAVE) {
            tape_st32(TL.a_rgb0, c0, hs0);
            mask_st(TL.m_rgb0, c0 >> 5, sign_word());
          }
        }
        if constexpr (SAVE) {  // raw view direction: the rgb.0 operand columns that stay in fp32 SIMT (bg fields)
          if (p.desc.L_dir == 0 && tape_tile != nullptr && TL.a_dir >= 0)
            *reinterpret_cast<uint4*>(tape_tile + tape_row_off(TL.n_a, TL.a_dir, row) + ((row & 7u) << 4)) =
                make_uint4(Op::pack2(dir_f.x, dir_f.y), Op::pack2(dir_f.z, 0.f), 0u, 0u);
        }
        a0 += lds32(sc_s + 4u * SC_RGB2_B0); a1 += lds32(sc_s + 4u * SC_RGB2_B1); a2 += lds32(sc_s + 4u * SC_RGB2_B2);
        st3(p.out.rgb, 1.f / (1.f + __expf(-a0)), 1.f / (1.f + __expf(-a1)), 1.f / (1.f + __expf(-a2)));
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();  // no CTA exits while its peer may still signal its barriers
  if (warp == 9) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <class Op, int B, int LMAX, bool DENSE, int WIDTH, bool SPLIT, bool SAVE>
static cudaError_t launch_one(const FieldKernelParams& p, int n_sm, cudaStream_t stream) {
  auto kern = field_fwd_kernel<Op, B, LMAX, DENSE, WIDTH, SPLIT, SAVE>;
  constexpr int kPer = SPLIT ? 1 : 2;  // tiles in flight per CTA
  const int smem = 1024 + kSmemArena + kSmemRing + (p.prog.cl.n_floats + kGroups * p.prog.fl.n_floats) * 4 + kBarBytes +
                   (SPLIT ? kSdfPartBytes : 0);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  int grid = (p.n_tiles + kPer - 1) / kPer < n_sm ? (p.n_tiles + kPer - 1) / kPer : n_sm;
  grid = (grid + kCluster - 1) / kCluster * kCluster;
  if (grid > n_sm) grid -= kCluster;
  if (grid < kCluster) grid = kCluster;
  if (grid > kMaxCtas) return cudaErrorInvalidValue;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // overlap the set-up with the prologue kernel's tail
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  return cudaLaunchKernelEx(&cfg, kern, p);
}

}  // namespace fwd

#ifndef B200R_SAVE
#define B200R_SAVE false
#endif
#if B200R_SAVE
cudaError_t launch_field_fwd_train(const FieldKernelParams& p, int n_sm, cudaStream_t stream) {
#else
cudaError_t launch_field_fwd(const FieldKernelParams& p, int n_sm, cudaStream_t stream) {
#endif
  const int od = p.desc.operand_dtype;
#define B200R_CASE(BN, LM, DN, WD)                                                                    \
  if (p.desc.n_bones == BN && p.Lmax == LM && (p.desc.dense != 0) == DN && p.desc.W == WD)            \
    return od == 1 ? fwd::launch_one<OpBF16, BN, LM, DN, WD, false, B200R_SAVE>(p, n_sm, stream)      \
                   : (od == 2 ? fwd::launch_one<OpF16, BN, LM, DN, WD, true, B200R_SAVE>(p, n_sm, stream) \
                              : fwd::launch_one<OpF16, BN, LM, DN, WD, false, B200R_SAVE>(p, n_sm, stream));
  B200R_CASE(0, 10, false, 128)
  B200R_CASE(0, 12, false, 128)
  B200R_CASE(0, 10, false, 256)
  B200R_CASE(0, 12, false, 256)
  B200R_CASE(18, 12, false, 256)
  B200R_CASE(25, 12, false, 256)
  B200R_CASE(18, 12, true, 256)
  B200R_CASE(25, 12, true, 256)
#undef B200R_CASE
  return cudaErrorInvalidValue;
}

}  // namespace b200r
