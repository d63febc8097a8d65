// bdiff_edge_tc.cuh — declarations of the tensor-core edge tile of the layer megakernel (bdiff_layers_tc.cu):
// tile / TMEM constants, shared-memory layout, weight-slab stream, the per-thread vector-channel update.
#pragma once
#include "bdiff_kernels.h"
#include "bdiff_slab.cuh"

namespace bdiff {

constexpr int TMT = 128;                 // edges per tile
// weight ring: TC_NSLOT slots of TC_SLOT bytes; a chunk is one slab plane (N rows x 32 B, N <= 320) or a group of
// small planes, always a single contiguous TMA bulk copy
constexpr int TC_SLOT = 2 * 160 * 32;    // 10 KiB: holds the widest chunk (9 KiB: a node-tile K step of 144 local rows, hi + lo)
constexpr int TC_NSLOT = 5;
// TMEM column map of an edge tile (512 columns allocated)
constexpr int TM_S = 0, TM_U0 = 256, TM_U1 = 288, TM_MV = 320, TM_VD0 = 416;
constexpr int TM_EX = 416, TM_EX_STRIDE = 40;     // pair-exchange scratch (over VD0, which is dead by then): 2 x 40 columns

__host__ __device__ constexpr int tc_k0_steps(int Ed, int Xd) {     // K=16 steps of message GCP 0's edge part
  return (Ed + (64 + Xd) / 4 + 9 + 15) / 16;
}
// bytes of one layer's edge-pass weight stream (see k_pack_edge_slabs for the order)
__host__ __device__ constexpr size_t tc_edge_stream_bytes(int Ed, int Xd) {
  return (size_t)tc_k0_steps(Ed, Xd) * 2 * 256 * 32 + 3 * ((size_t)16 * 2 * 320 * 32 + 2 * 2 * 256 * 32) + (size_t)16 * 2 * 32 * 32;
}

// One CTA's half of an edge tile's weight stream as TMA chunks (one bulk copy and one ring slot each), in issue order:
//   G0                      k0s chunks: one K step of 128 rows ([hi plane | lo plane])
//   k = 1..3   U pass         4 chunks: 4 K steps of the 32 gate rows each
//              S pass        16 chunks: one K step of 128 rows of W_k
//              G(k)b          2 chunks: one K step of 128 rows (W_k K rows 256..287)
//   G4                        4 chunks: 4 K steps of 16 rows of Wg_3 each
// The TMA producer streams exactly these chunks and the peer's relay lane forwards one completion per chunk, so both
// take their count from here.
constexpr uint32_t TC_EC_S = 2 * 128 * 32, TC_EC_U = 4 * 2 * 32 * 32, TC_EC_G4 = 4 * 2 * 16 * 32;
constexpr int TC_EC_PER_GCP = 4 + 16 + 2;
__host__ __device__ constexpr int tc_edge_tile_chunks(int k0s) { return k0s + 3 * TC_EC_PER_GCP + 4; }
__host__ __device__ constexpr uint32_t tc_edge_chunk_bytes(int k0s, int c) {
  return c < k0s ? TC_EC_S : c < k0s + 3 * TC_EC_PER_GCP ? ((c - k0s) % TC_EC_PER_GCP < 4 ? TC_EC_U : TC_EC_S) : TC_EC_G4;
}
__host__ __device__ constexpr size_t tc_edge_chunks_total_bytes(int k0s) {     // both CTAs
  size_t b = 0;
  for (int c = 0; c < tc_edge_tile_chunks(k0s); ++c) b += tc_edge_chunk_bytes(k0s, c);
  return 2 * b;
}
static_assert(tc_edge_chunks_total_bytes(tc_k0_steps(64, 16)) == tc_edge_stream_bytes(64, 16) &&
              tc_edge_chunks_total_bytes(tc_k0_steps(16, 8)) == tc_edge_stream_bytes(16, 8),
              "edge chunk table and packed stream size disagree");
static_assert(TC_EC_S <= TC_SLOT && TC_EC_U <= TC_SLOT && TC_EC_G4 <= TC_SLOT, "an edge chunk fits one ring slot");

// mbarriers / bookkeeping of the megakernel; first member (base class) of both tile tails.  u_full: the gate pass of an
// edge GCP is complete (its own commit, ahead of the S pass that d_full waits for).
struct TcBars {
  uint64_t full[TC_NSLOT], empty[TC_NSLOT], pfull[TC_NSLOT], a_ready, d_full, wbar, u_free, u_full;
  uint64_t item_full[2], item_empty[2], peer_empty[2], tile_done;
  alignas(16) int item[2][4];   // work items {type, layer, tile of THIS CTA, -}; the leader writes the peer's copy (16-byte st.shared::cluster)
  uint32_t tmem_ptr;
  uint32_t pad_;
};

// Thread roles: warps 0-7 epilogue/compute — edge r of the tile is owned by the thread PAIR (r, r+128): "half" 0
// works on accumulator columns [0,128) and vector channels [0,16), half 1 on columns [128,256) and channels
// [16,32) (both warps of a pair address the same TMEM lanes: lane quarter = warp % 4); warp 8 = scheduler + TMA
// producer (+ TMEM allocator), warp 9 = MMA issuer.
constexpr int TC_EPI = 256;

struct alignas(16) SmallW {   // fp32 copies of the thread-local (vector channel) weights, broadcast-read
  float Wd0x[16 * 20];     // [Xd][hid0]
  float Wf0x[16 * 3];      // [Xd][3]
  float Wu0[20 * 32];      // [hid0][32]
  float Wdk[3][32 * 8];    // [32][8]
  float Wfk[3][32 * 3];    // [32][3]
  float Wuk[3][8 * 32];    // [8][32]
  float bg[4][32];
  float bk[3][256];
  float wa[256];
  float ba[4];
};

struct EdgeTail : TcBars {
  float2 wbuf[2][8][2][32];   // [round parity][16-row window]: [0] head piece (segment entered from the previous window), [1] tail / whole piece
  SmallW sw;
  float sAttn[2][TMT];
  int sRow[TMT], sCol[TMT], sB[TMT], sNa[TMT];
  uint32_t winfo[8];       // per window: start mask | end mask << 16
};

// Gate of the previous GCP from TMEM (U), vector-message update in TMEM scratch for this thread's 16 channels,
// and this thread's partial vector_down / vector_down_frames sums of the NEXT GCP.
// HP = hidden dim of the previous GCP; vdp = its vector_down output (full, [HP][3]).
template <int HP, bool FIRST, bool LAST>
__device__ __forceinline__ void gate_update(uint32_t tl, int half, int ucol, const float* __restrict__ vdp,
                                            const float* __restrict__ Wu, const float* __restrict__ bgp,
                                            const float* __restrict__ Wdn, const float* __restrict__ Wfn,
                                            float* __restrict__ part) {   // part[33]: partial VD_next(24)+VDF_next(9)
  float2 p2[4][3];                 // VD_next accumulators, pairs of hidden rows (h = 2hp, 2hp+1) per component
  if (!LAST) {
#pragma unroll
    for (int i = 0; i < 33; ++i) part[i] = 0.f;
#pragma unroll
    for (int hp = 0; hp < 4; ++hp) { p2[hp][0] = make_float2(0.f, 0.f); p2[hp][1] = p2[hp][0]; p2[hp][2] = p2[hp][0]; }
  }
  for (int oc = half * 2; oc < half * 2 + 2; ++oc) {
    float u[8], mv[24];
    {
      uint32_t ru[8], rm[24];
      tmem_ld8_nw(tl + ucol + oc * 8, ru);
      if (!FIRST) {
        tmem_ld8_nw(tl + TM_MV + oc * 24, rm);
        tmem_ld8_nw(tl + TM_MV + oc * 24 + 8, rm + 8);
        tmem_ld8_nw(tl + TM_MV + oc * 24 + 16, rm + 16);
      }
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 8; ++i) u[i] = __uint_as_float(ru[i]);
      if (!FIRST) {
#pragma unroll
        for (int i = 0; i < 24; ++i) mv[i] = __uint_as_float(rm[i]);
      }
    }
#pragma unroll
    for (int jp = 0; jp < 4; ++jp) {          // two output channels (j = 2jp, 2jp+1) per packed instruction
      const int o = oc * 8 + 2 * jp;
      const float2 g = sigmoid_acc2(__fadd2_rn(make_float2(u[2 * jp], u[2 * jp + 1]),
                                               *reinterpret_cast<const float2*>(bgp + o)));
      float2 s0 = make_float2(0.f, 0.f), s1 = s0, s2 = s0;
#pragma unroll
      for (int h = 0; h < HP; ++h) {
        const float2 wu = *reinterpret_cast<const float2*>(Wu + h * 32 + o);
        s0 = __ffma2_rn(wu, make_float2(vdp[h * 3 + 0], vdp[h * 3 + 0]), s0);
        s1 = __ffma2_rn(wu, make_float2(vdp[h * 3 + 1], vdp[h * 3 + 1]), s1);
        s2 = __ffma2_rn(wu, make_float2(vdp[h * 3 + 2], vdp[h * 3 + 2]), s2);
      }
      const int ja = 2 * jp * 3, jb = (2 * jp + 1) * 3;
      float2 r0, r1, r2;
      if (FIRST) { r0 = __fmul2_rn(s0, g); r1 = __fmul2_rn(s1, g); r2 = __fmul2_rn(s2, g); }
      else {
        r0 = __ffma2_rn(s0, g, make_float2(mv[ja + 0], mv[jb + 0]));
        r1 = __ffma2_rn(s1, g, make_float2(mv[ja + 1], mv[jb + 1]));
        r2 = __ffma2_rn(s2, g, make_float2(mv[ja + 2], mv[jb + 2]));
      }
      mv[ja + 0] = r0.x; mv[jb + 0] = r0.y; mv[ja + 1] = r1.x; mv[jb + 1] = r1.y; mv[ja + 2] = r2.x; mv[jb + 2] = r2.y;
    }
    tmem_st8xN<3>(tl + TM_MV + oc * 24, mv);      // completion awaited once, at the end of the function
    if (!LAST) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = oc * 8 + j;
        const float4 wd0 = *reinterpret_cast<const float4*>(Wdn + c * 8), wd1 = *reinterpret_cast<const float4*>(Wdn + c * 8 + 4);
        const float2 wdp[4] = {make_float2(wd0.x, wd0.y), make_float2(wd0.z, wd0.w), make_float2(wd1.x, wd1.y),
                               make_float2(wd1.z, wd1.w)};
#pragma unroll
        for (int x = 0; x < 3; ++x) {
          const float2 mb = make_float2(mv[j * 3 + x], mv[j * 3 + x]);
#pragma unroll
          for (int hp = 0; hp < 4; ++hp) p2[hp][x] = __ffma2_rn(wdp[hp], mb, p2[hp][x]);
        }
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          const float wf = Wfn[c * 3 + ch];
          part[24 + ch * 3 + 0] = fmaf(wf, mv[j * 3 + 0], part[24 + ch * 3 + 0]);
          part[24 + ch * 3 + 1] = fmaf(wf, mv[j * 3 + 1], part[24 + ch * 3 + 1]);
          part[24 + ch * 3 + 2] = fmaf(wf, mv[j * 3 + 2], part[24 + ch * 3 + 2]);
        }
      }
    }
  }
  if (!LAST) {
#pragma unroll
    for (int hp = 0; hp < 4; ++hp)
#pragma unroll
      for (int x = 0; x < 3; ++x) { part[(2 * hp) * 3 + x] = p2[hp][x].x; part[(2 * hp + 1) * 3 + x] = p2[hp][x].y; }
  }
  tmem_st_wait();
}

// The two threads of a pair (same TMEM lane) swap their 33 partial sums through TMEM scratch columns: no shared memory.
// Callers guarantee that nobody still reads the columns (VD0) being overwritten.
__device__ __forceinline__ void pair_exchange33(uint32_t tl, int half, const float* __restrict__ mine, float* __restrict__ theirs) {
  float pad[40];
#pragma unroll
  for (int i = 0; i < 33; ++i) pad[i] = mine[i];
#pragma unroll
  for (int i = 33; i < 40; ++i) pad[i] = 0.f;
  tmem_st8xN<5>(tl + TM_EX + half * TM_EX_STRIDE, pad);
  tmem_st_wait();
  tc_fence_before();
  named_bar_sync(3, TC_EPI);
  tc_fence_after();
  float got[40];
  tmem_ld8xN<5>(tl + TM_EX + (half ^ 1) * TM_EX_STRIDE, got);
#pragma unroll
  for (int i = 0; i < 33; ++i) theirs[i] = got[i];
}

}  // namespace bdiff
