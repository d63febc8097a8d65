// bdiff_layers_tc.cu — all L interaction layers of one denoiser forward in ONE persistent tensor-core kernel.
//
// Why: with one kernel per pass the forward is quantised twice per layer — 361 edge tiles on 148 SMs are three
// rounds (19 % of the SM time idle in the last one at the BASELINE batch) and the node pass has work for only 76
// SMs — and pays ~18 launch / prologue / pipeline-ramp gaps.  Nothing in the network couples molecules inside a
// layer (gcpnet.py:676-737, 893-930: messages, aggregation and node updates are per molecule), so layer l+1 of
// a molecule only needs layer l of the same molecule.  This kernel therefore runs the edge-tile and node-tile bodies
// (edge_tile_*.inc, node_r4_tile_*.inc) from a global work list of tile PAIRS (see below)
//     for l in 0..L-1:  edge pairs (l, 0..PE-1) in order, node pair (l, v) inserted ~one wave of claims after the last
//                       edge pair it depends on (so its wait is short and the CTA pair that claims it does not idle)
// claimed with one atomicAdd per item, with per-tile completion flags as dependencies:
//     edge (l, t)  waits for node (l-1, u) of every 32-node tile u that intersects the molecules of edge tile t;
//     node (l, u)  waits for edge (l, t) of every edge tile t that intersects the molecules of node tile u.
// Every dependency has a smaller queue index and a pair only claims an item once it is running, so the smallest unfinished
// item can always run: no deadlock.  A dependency wait beyond 2^32 cycles can only mean a broken schedule: it traps (sticky
// launch failure + error word read by bdiff_check) instead of computing on stale data.
// Flags are released with fence + st.release after a CTA barrier and acquired with ld.acquire + a gpu-scope fence
// in every consumer thread (mutable activations are re-read from L2, not from a stale L1 line).
//
// The TMA-producer lane also claims the items (so the next tile's weights stream while the current tile computes) and hands
// them to the MMA lane and the 8 compute warps through a two-slot mbarrier ring.
#include "bdiff_node_tc.cuh"

namespace bdiff {

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Shared memory: [A region: 9 x 16 KiB (edge tile: hi blocks 0-3, lo blocks 4-7, extra block 8; node tile: 5 R5 blocks
// of 20 KiB + NodeScratch)] [weight ring: TC_NSLOT x 10 KiB] [tail: barriers + per-tile small weights / buffers].
union LayersTail {
  TcBars bars;
  EdgeTail edge;
  NodeTail node;
};
constexpr size_t LAYERS_SMEM_BYTES = XE_BLOCKS * (size_t)X_BLOCK + TC_NSLOT * (size_t)TC_SLOT + sizeof(LayersTail) + 1024;
static_assert(LAYERS_SMEM_BYTES <= 232448, "shared memory budget of the layer megakernel");

// The grid is a set of CTA PAIRS (thread-block clusters of 2, cta_group::2): a pair works on two consecutive tiles of the same
// kind and layer at a time (CTA rank r on tile 2j + r), ONE thread of the leader CTA (rank 0) issues every MMA for both SMs
// (M = 256: each CTA's own A tile and TMEM), and every weight plane is SPLIT between the two shared memories, so each SM
// streams, stores and reads only half of the weights: 2.3 GB of L2->SM weight traffic per QM9 forward instead of 4.6 GB and
// 49 KB instead of 74 KB of shared-memory traffic per K step.  Cross-CTA protocol: events are forwarded to the leader by single
// RELAXED remote mbarrier arrives — the peer's operand publications / U releases by a relay lane (warp 10), its TMA
// completions by one relay lane per ring slot (warp 9); the leader's commits are multicast to both CTAs (ring slots, d_full);
// work items are claimed by the leader's scheduler lane and handed to the peer through distributed shared memory.
// (Measured: same speed as the single-CTA version — 60.9 vs 61.2 molecules/s — the MMA phases are bound by the
// instruction mix (N=64 / N=32 MMAs at ~50 cycles, per-K-step bookkeeping of the issuing lane), not by operand bandwidth.)
//
// 12 warps: 0-7 compute (two warpgroups), 8 scheduler + TMA producer, 9 MMA issuer, 10-11 padding so that the
// service warps form a complete third warpgroup for setmaxnreg.  The CTA is launched with 168 registers/thread
// (384 threads -> a pool of 64512); the service warpgroup shrinks to 96 and the two compute warpgroups grow to 200
// (256*200 + 128*96 = 63488 <= 64512 — a request the pool cannot satisfy would block forever).
constexpr int LAYERS_THREADS = 384;
constexpr int LAYERS_REG_COMPUTE = 200, LAYERS_REG_SERVICE = 96;
static_assert(256 * LAYERS_REG_COMPUTE + 128 * LAYERS_REG_SERVICE <= 168 * LAYERS_THREADS, "setmaxnreg pool");

// acquire at cluster scope: the item slot / remote arrivals come from the other CTA of the pair
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void st_cluster_v4(uint32_t cluster_addr, int a, int b, int c, int d) {
  asm volatile("st.shared::cluster.v4.s32 [%0], {%1, %2, %3, %4};" ::"r"(cluster_addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

template <int ED, int XD>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(LAYERS_THREADS, 1)
    k_layers_tc(Plan p, Dims d, EmbedW ew, LayerSched q, Work w) {
  constexpr int HID0 = (64 + XD) / 4;
  constexpr int H2 = HID0 / 2;
  constexpr int K0RAW = ED + HID0 + 9;
  constexpr int K0S = (K0RAW + 15) / 16;
  static_assert(HID0 % 2 == 0 && H2 * 3 <= 32 && HID0 + 9 <= 32 && ED % 16 == 0, "layout");

  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* X = smem;
  unsigned char* ring = smem + XE_BLOCKS * X_BLOCK;
  unsigned char* tail = ring + TC_NSLOT * TC_SLOT;
  TcBars& B = *reinterpret_cast<TcBars*>(tail);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int hid0 = d.hid0;
  const int per_layer = q.TE + q.TN;
  const int total_items = q.nitems;                 // pair items
  int* const flags = q.sched + 2;
  const uint32_t rank = cluster_ctarank();          // 0 = leader of the pair
  const bool leader = rank == 0;

  if (tid == 0) {
    for (int i = 0; i < TC_NSLOT; ++i) { mbar_init(&B.full[i], 1); mbar_init(&B.empty[i], 1); mbar_init(&B.pfull[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&B.item_full[i], 1); mbar_init(&B.item_empty[i], leader ? TC_EPI + 1 : TC_EPI + 2); mbar_init(&B.peer_empty[i], 1);
    }
    mbar_init(&B.tile_done, TC_EPI);
    mbar_init(&B.a_ready, leader ? TC_EPI + 1 : TC_EPI);   // leader's: its own compute threads + ONE arrival relayed by the peer's MMA lane
    mbar_init(&B.d_full, 1);
    mbar_init(&B.u_full, 1);
    mbar_init(&B.wbar, 1);
    mbar_init(&B.u_free, leader ? TC_EPI + 1 : TC_EPI);
    mbar_fence_init();
  }
  cluster_sync_all();                               // the barriers of both CTAs exist before any remote arrive
  if (warp == 8) tmem_alloc2(&B.tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = B.tmem_ptr;
  // Cross-CTA events are forwarded by ONE relaxed remote arrive of the peer's MMA lane (an arrive.release.cluster costs the
  // issuing thread ~800 cycles of fencing, and 256 of them per phase — or one per weight plane — made the first pair version
  // slower than the single-CTA kernel).  The data itself never crosses SMs: every tensor core reads its own SM's shared memory.
  const uint32_t a_ready_leader = mapa_u32(&B.a_ready, 0), u_free_leader = mapa_u32(&B.u_free, 0);

  if (warp == 8) {
    // ============================================================ scheduler + TMA producer (one lane)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(LAYERS_REG_SERVICE));
    if (lane == 0) {
      uint32_t ci = 0;
      for (uint32_t k = 0;; ++k) {
        const uint32_t slot = k & 1;
        mbar_wait_backoff(&B.item_empty[slot], ((k >> 1) & 1) ^ 1);
        int type = -1, layer = 0, tile = 0;
        if (leader) {
          // the peer's copy of this item slot is free as well (its scheduler lane relays its item_empty)
          mbar_wait_backoff(&B.peer_empty[slot], (k >> 1) & 1);
          const int qi = atomicAdd(q.sched, 1);
          int pair = 0;
          if (qi < total_items) {
            const int it = __ldg(q.items + qi);
            type = (it >> 30) & 1; layer = (it >> 24) & 63; pair = it & 0xffffff;
          }
          B.item[slot][0] = type; B.item[slot][1] = layer; B.item[slot][2] = 2 * pair;
          st_cluster_v4(mapa_u32(&B.item[slot][0], 1), type, layer, 2 * pair + 1, 0);
          mbar_arrive(&B.item_full[slot]);
          mbar_arrive_remote(mapa_u32(&B.item_full[slot], 1));      // release.cluster: the item words are visible to the peer
          tile = 2 * pair;
        } else {
          mbar_arrive_remote_relaxed(mapa_u32(&B.peer_empty[slot], 0));
          mbar_wait_cluster(&B.item_full[slot], (k >> 1) & 1);
          type = B.item[slot][0]; layer = B.item[slot][1]; tile = B.item[slot][2];
        }
        (void)tile;
        if (type < 0) break;
        // this CTA's half of the layer's weight stream: [rank 0 stream | rank 1 stream]
        const unsigned char* blob = type == 0 ? q.edge_blob + (size_t)layer * q.edge_blob_stride + rank * (q.edge_blob_stride / 2)
                                              : q.node_blob + (size_t)layer * q.node_blob_stride + rank * (q.node_blob_stride / 2);
        size_t off = 0;
        auto push = [&](uint32_t bytes) {
          const uint32_t s = ci % TC_NSLOT;
          mbar_wait_backoff(&B.empty[s], ((ci / TC_NSLOT) & 1) ^ 1);
          mbar_expect_tx(&B.full[s], bytes);
          bulk_g2s(ring + s * TC_SLOT, blob + off, bytes, &B.full[s]);
          off += bytes;
          ++ci;
        };
        if (type == 0) {
#include "edge_tile_producer.inc"
        } else {
          const int last = layer == q.L - 1;
#include "node_r4_tile_producer.inc"
        }
      }
    }
  } else if (warp == 9 && !leader) {
    // ============ peer: its weight planes are consumed by MMAs the LEADER issues, so their TMA completions (local full barriers)
    // are forwarded to the leader's pfull barriers.  A remote arrive keeps the issuing thread busy for ~600 cycles: one lane per
    // ring slot shares the work.  Lane 0 also publishes the completion flag of the peer's tile.
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(LAYERS_REG_SERVICE));
    if (lane < TC_NSLOT) {
      const uint32_t pfull0 = mapa_u32(&B.pfull[0], 0);
      uint32_t ci = 0;
      for (uint32_t k = 0;; ++k) {
        const uint32_t slot = k & 1;
        mbar_wait_cluster(&B.item_full[slot], (k >> 1) & 1);
        const int type = B.item[slot][0], layer = B.item[slot][1], tile = B.item[slot][2];
        if (type < 0) break;
        const uint32_t nch = type == 0 ? (uint32_t)tc_edge_tile_chunks(K0S) : (layer == q.L - 1 ? 73u : 100u);   // chunks per tile (producer includes)
        // lane = ring slot: a lane sees the phases of ITS slot's barrier strictly in order (waiting for a phase two uses ahead
        // would alias with the parity of the current one)
        for (uint32_t cc = ci + ((lane + TC_NSLOT - ci % TC_NSLOT) % TC_NSLOT); cc < ci + nch; cc += TC_NSLOT) {
          mbar_wait_backoff(&B.full[lane], (cc / TC_NSLOT) & 1);
          mbar_arrive_remote_relaxed(pfull0 + lane * 8);
        }
        ci += nch;
        if (lane == 0) {
          mbar_wait_backoff(&B.tile_done, k & 1);
          __threadfence();
          if (tile < (type == 0 ? q.TE : q.TN))
            st_release_gpu(flags + (size_t)layer * per_layer + (type == 0 ? tile : q.TE + tile), 1);
          mbar_arrive(&B.item_empty[slot]);
        }
      }
    }
  } else if (warp == 9) {
    // =============================== leader: MMA lane, issues every pair MMA (cta_group::2) for both CTAs
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(LAYERS_REG_SERVICE));
    if (lane == 0) {
      TcBars& T = B;
      const uint32_t i256 = umma_idesc_bf16_m256(256), i64 = umma_idesc_bf16_m256(64), i32 = umma_idesc_bf16_m256(32);
      const uint32_t xaddr = smem_u32(X), raddr = smem_u32(ring);
      uint32_t ci = 0, pa = 0, pu = 0;
      long long wcyc = 0, acyc = 0;          // BDIFF_TIMING: cycles this lane spent waiting for weights / for operands
      auto wait_a = [&]() {
        if (!leader) return;                                   // the peer's operands are announced by its relay lane (warp 10)
        const long long t0 = w.dbg ? clock64() : 0;
        mbar_wait_backoff(&B.a_ready, pa); pa ^= 1;
        tc_fence_after();
        if (w.dbg) acyc += clock64() - t0;
      };
      // leader: both halves of the plane have landed (mine: full, the peer's: pfull, relayed);  peer: relay, no MMAs
      auto wait_w = [&]() -> uint32_t {
        const uint32_t s = ci % TC_NSLOT, par = (ci / TC_NSLOT) & 1;
        const long long t0 = w.dbg ? clock64() : 0;
        mbar_wait_backoff(&B.full[s], par);
        mbar_wait_backoff(&B.pfull[s], par);
        if (w.dbg) wcyc += clock64() - t0;
        return raddr + s * TC_SLOT;
      };
      auto done_w = [&]() { if (leader) umma_commit_pair(&B.empty[ci % TC_NSLOT]); ++ci; };
      auto commit_d = [&]() { if (leader) umma_commit_pair(&B.d_full); };
      auto commit_u = [&]() { if (leader) umma_commit_pair(&B.u_full); };
      auto mma = [&](uint32_t dcol, uint64_t ad, uint64_t bd, uint32_t idesc, bool acc) { if (leader) umma_bf16_pair(tmem + dcol, ad, bd, idesc, acc); };
      // node-tile GEMMs over A blocks 0..3 (R5 layout: views at row 0 and row 32, four products per K step).  Local plane =
      // [128 rows of the S columns | 16 gate rows] (NL rows): S is one N=256 pair MMA, the gate accumulator U (columns 256..287)
      // one N=32 pair MMA: umode 1 accumulates +Wg h_new, umode 2 starts U = -Wg h_old (sign folded into the packed weights).
      auto ngemm = [&](int NL, uint32_t dcol, bool fresh, int umode) {
        for (int ks = 0; ks < 16; ++ks) {
          const uint32_t a = xaddr + (ks >> 2) * R5_BLOCK + (ks & 3) * 32;
          const uint64_t v0 = umma_desc_sw128(a), v1 = umma_desc_sw128(a + 4096);
          const uint32_t wb0 = wait_w();                      // one chunk = this K step's [hi plane | lo plane]
          for (int pl = 0; pl < 2; ++pl) {
            const uint32_t wb = wb0 + pl * NL * 32;
            const bool first = ks == 0 && pl == 0;
            const uint64_t bs = umma_desc_k16(wb, NL * 16, 128);
            mma(dcol, v0, bs, i256, fresh ? !first : true);
            mma(dcol, v1, bs, i256, true);
            if (umode) {
              const uint64_t bu = umma_desc_k16(wb + 128 * 16, NL * 16, 128);
              mma(NM_U, v0, bu, i32, umode == 2 ? !first : true);
              mma(NM_U, v1, bu, i32, true);
            }
          }
          done_w();
        }
      };
      auto nextra = [&]() {                                  // += [vn | q] (block 4, 32 columns) . W[:, 256:288]
        for (int ks = 0; ks < 2; ++ks) {
          const uint32_t a = xaddr + 4 * R5_BLOCK + ks * 32;
          const uint64_t v0 = umma_desc_sw128(a), v1 = umma_desc_sw128(a + 4096);
          const uint32_t wb0 = wait_w();
          for (int pl = 0; pl < 2; ++pl) {
            const uint32_t wb = wb0 + pl * 128 * 32;
            mma(NM_S, v0, umma_desc_k16(wb, 128 * 16, 128), i256, true);
            mma(NM_S, v1, umma_desc_k16(wb, 128 * 16, 128), i256, true);
          }
          done_w();
        }
      };
      for (uint32_t k = 0;; ++k) {
        const uint32_t slot = k & 1;
        mbar_wait_cluster(&B.item_full[slot], (k >> 1) & 1);
        const int type = B.item[slot][0], layer = B.item[slot][1], tile = B.item[slot][2];
        if (type < 0) break;
        const long long tstart = w.dbg ? clock64() : 0;
        wcyc = 0; acyc = 0;
        if (type == 0) {
#include "edge_tile_mma.inc"
        } else {
          const int last = layer == q.L - 1;
#include "node_r4_tile_mma.inc"
        }
        if (w.dbg && k >= 2 && k < 4) {     // items 2, 3 of this CTA: {item code, total cycles, weight-wait, operand-wait}
          long long* o = w.dbg + 256 * 64 + 148 * 64 + (size_t)blockIdx.x * 8 + (k - 2) * 4;
          o[0] = (type << 30) | (layer << 24) | tile; o[1] = clock64() - tstart; o[2] = wcyc; o[3] = acyc;
        }
        mbar_wait_backoff(&B.tile_done, k & 1);
        __threadfence();
        if (tile < (type == 0 ? q.TE : q.TN))       // a ghost tile (odd tile count) has no flag
          st_release_gpu(flags + (size_t)layer * per_layer + (type == 0 ? tile : q.TE + tile), 1);
        mbar_arrive(&B.item_empty[slot]);
      }
    }
  } else if (warp == 10) {
    // ============ peer only: event relay lane.  It waits on the peer's LOCAL a_ready / u_free (the peer's 256 compute threads)
    // and forwards each completion to the leader's barrier with one relaxed remote arrive.
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(LAYERS_REG_SERVICE));
    if (lane == 0 && !leader) {
      uint32_t pa = 0, pu = 0;
      for (uint32_t k = 0;; ++k) {
        const uint32_t slot = k & 1;
        mbar_wait_cluster(&B.item_full[slot], (k >> 1) & 1);
        const int type = B.item[slot][0], layer = B.item[slot][1];
        if (type < 0) break;
        const bool has_u = type == 1 && layer != q.L - 1;
        const int nph = type == 0 ? 8 : 6;                      // operand publications per tile (edge: G0, 3 x (a, b), G4)
        for (int ph = 0; ph < nph; ++ph) {
          if (has_u && ph == 4) { mbar_wait_backoff(&B.u_free, pu); pu ^= 1; mbar_arrive_remote_relaxed(u_free_leader); }
          mbar_wait_backoff(&B.a_ready, pa); pa ^= 1;
          mbar_arrive_remote_relaxed(a_ready_leader);
        }
        mbar_arrive(&B.item_empty[slot]);
      }
    }
  } else if (warp >= 11) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(LAYERS_REG_SERVICE));     // padding warp of the service warpgroup
  } else {
    // ============================================================================ compute / epilogue warps
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(LAYERS_REG_COMPUTE));
    uint32_t pd = 0, pg = 0, pw = 0;
    int cur_type = -1, cur_layer = -1;
    // BDIFF_TIMING: phase stamps (clock64) of the first edge / node item with k >= 2 of every CTA: [128 + 0..31] edge,
    // [128 + 32..63] node — one stamp before and after every accumulator wait, one after every operand publication
    int es = 0;
    long long* stamp = nullptr;
    auto PH = [&]() { if (stamp && tid == 0 && es < 32) stamp[es] = clock64(); ++es; };
    auto wait_d = [&]() { PH(); mbar_wait(&B.d_full, pd); pd ^= 1; tc_fence_after(); PH(); };
    auto wait_u = [&]() { PH(); mbar_wait(&B.u_full, pg); pg ^= 1; tc_fence_after(); PH(); };     // edge tiles: gate pass done
    auto publish = [&]() { fence_proxy_async(); tc_fence_before(); mbar_arrive(&B.a_ready); PH(); };
    bool stamped[2] = {false, false};
    const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    auto sz = [](int n) { return (uint32_t)((n * 4 + 15) & ~15); };
    for (uint32_t k = 0;; ++k) {
      const uint32_t slot = k & 1;
      mbar_wait_cluster(&B.item_full[slot], (k >> 1) & 1);
      const int type = B.item[slot][0], layer = B.item[slot][1], tile = B.item[slot][2];
      if (type < 0) break;
      const bool real = tile < (type == 0 ? q.TE : q.TN);      // odd tile counts: the last pair's second CTA runs a ghost tile
      if (tid == 0 && w.dbg && k < 16) {      // BDIFF_TIMING: {item code, t_fetch, t_start, t_end} for the first 16 items
        w.dbg[(size_t)blockIdx.x * 64 + 4 * k] = (type << 30) | (layer << 24) | tile;
        w.dbg[(size_t)blockIdx.x * 64 + 4 * k + 1] = clock64();
      }
      // ---- small (vector-channel) weights of this (pass, layer): reload only when they change
      if (type != cur_type || layer != cur_layer) {
        named_bar_sync(3, TC_EPI);             // everybody is done with the previous set
        if (tid == 0) {
          const LayerW lw = q.layers[layer];       // by value: the pointer loads go out together, not one per copy
          if (type == 0) {
            SmallW& s = reinterpret_cast<EdgeTail*>(tail)->sw;
            mbar_expect_tx(&B.wbar, sz(XD * HID0) + sz(XD * 3) + sz(HID0 * 32) +
                                        3 * (sz(256) + sz(256) + sz(256) + sz(96) + sz(32)) + sz(32) + sz(256) + sz(1));
            auto cp = [&](float* dst, const float* src, int n) { bulk_g2s(dst, src, sz(n), &B.wbar); };
            cp(s.Wd0x, lw.Wd0x, XD * HID0); cp(s.Wf0x, lw.Wf0x, XD * 3); cp(s.Wu0, lw.Wu0, HID0 * 32);
            for (int kk = 0; kk < 3; ++kk) {
              cp(s.Wdk[kk], lw.Wdk[kk], 256); cp(s.Wuk[kk], lw.Wuk[kk], 256); cp(s.bk[kk], lw.bk[kk], 256);
              cp(s.Wfk[kk], lw.Wfk[kk], 96); cp(s.bg[kk + 1], lw.bgk[kk], 32);
            }
            cp(s.bg[0], lw.bg0, 32); cp(s.wa, lw.wa, 256); cp(s.ba, lw.ba, 1);
          } else {
            const int last = layer == q.L - 1;
            const LayerW wn = q.layers[last ? layer : layer + 1];
            SmallWR4& s = reinterpret_cast<NodeTail*>(tail)->sw;
            uint32_t total = sz(1024) + sz(192) + sz(512) + sz(32) + 2 * sz(256) + sz(256) + sz(96) + sz(8) + 2 * sz(256) + sz(1);
            total += last ? sz(1024) + sz(96) + sz(d.Hin) : sz(256) + 2 * sz(32 * hid0) + 2 * sz(96);
            mbar_expect_tx(&B.wbar, total);
            auto cp = [&](float* dst, const float* src, int n) { bulk_g2s(dst, src, sz(n), &B.wbar); };
            cp(s.Wdf, lw.Wdf, 64 * 16); cp(s.Wff, lw.Wff, 64 * 3); cp(s.Wuf, lw.Wuf, 16 * 32); cp(s.bgf, lw.bgf, 32);
            cp(s.b1, lw.b1, 256); cp(s.b2, lw.b2, 256);
            cp(s.Wdp, lw.Wdp, 32 * 8); cp(s.Wfp, lw.Wfp, 32 * 3); cp(s.Wup, lw.Wup, 8); cp(s.bp, lw.bp, 256);
            cp(s.wgp, lw.Wgp, 256); cp(s.bgp, lw.bgp, 1);
            if (!last) {
              cp(s.u.nx.b0, wn.b0, 256);
              cp(s.u.nx.Wd0i, wn.Wd0i, 32 * hid0); cp(s.u.nx.Wd0j, wn.Wd0j, 32 * hid0);
              cp(s.u.nx.Wf0i, wn.Wf0i, 96); cp(s.u.nx.Wf0j, wn.Wf0j, 96);
            } else {
              cp(s.u.pj.pWd, ew.pWd, 32 * 32); cp(s.u.pj.pWf, ew.pWf, 96); cp(s.u.pj.pbs, ew.pbs, d.Hin);
            }
          }
        }
        mbar_wait(&B.wbar, pw);
        pw ^= 1;
        cur_type = type; cur_layer = layer;
      }
      // ---- dependencies: completion flags of the producer tiles (bounded spin), then a gpu-scope acquire in
      //      every thread before it reads activations written by other SMs
      if (tid == 0 && real) {
        int lo = 0, hi = -1;
        const int* fbase = flags;
        if (type == 0) {
          if (layer > 0) {
            const int2 dep = q.edge_dep[tile];
            lo = dep.x; hi = dep.y;
            fbase = flags + (size_t)(layer - 1) * per_layer + q.TE;
          }
        } else {
          const int2 dep = q.node_dep[tile];
          lo = dep.x; hi = dep.y;
          fbase = flags + (size_t)layer * per_layer;
        }
        const long long t0 = clock64();
        for (int u = lo; u <= hi; ++u) {
          while (ld_acquire_gpu(fbase + u) == 0) {
            // every producer precedes its consumer in the claim order and all CTAs are resident, so this wait is bounded
            // by a few tile times; > 2^32 cycles (~2 s) can only mean a broken schedule: record it and abort the kernel
            // HERE (sticky launch failure) rather than computing on stale data
            if (clock64() - t0 > (1ll << 32)) { atomicExch(q.err, 1); __threadfence_system(); __trap(); }
          }
        }
      }
      named_bar_sync(3, TC_EPI);
      __threadfence();
      if (tid == 0 && w.dbg && k < 16) w.dbg[(size_t)blockIdx.x * 64 + 4 * k + 2] = clock64();
      es = 0;
      stamp = nullptr;
      if (w.dbg && k >= 2 && !stamped[type]) { stamp = w.dbg + 256 * 64 + (size_t)blockIdx.x * 64 + type * 32; stamped[type] = true; }
      PH();
      if (type == 0) {
        EdgeTail& T = *reinterpret_cast<EdgeTail*>(tail);
        const int half = tid >> 7, r = tid & 127;
        const SmallW& sw = T.sw;
#include "edge_tile_epilogue.inc"
      } else {
        NodeTail& T = *reinterpret_cast<NodeTail*>(tail);
        NodeScratch& SC = *reinterpret_cast<NodeScratch*>(X + R5_BLOCKS * R5_BLOCK);
        const int last = layer == q.L - 1;
        const int l = lane, s = warp, c0 = warp * 32;
        const SmallWR4& sw = T.sw;
#include "node_r4_tile_epilogue.inc"
      }
      // ---- completion: every compute thread arrives (release) on tile_done after its last global write; the MMA
      //      lane — idle at this point — acquires it, makes the writes visible gpu-wide and raises the flag, so the
      //      ~1 us fence is off the compute warps' critical path
      PH();
      if (tid == 0 && w.dbg && k < 16) w.dbg[(size_t)blockIdx.x * 64 + 4 * k + 3] = clock64();
      mbar_arrive(&B.tile_done);
      mbar_arrive(&B.item_empty[slot]);
    }
    tc_fence_before();
  }
  __syncthreads();
  cluster_sync_all();                               // nobody leaves while the pair's barriers / TMEM may still be addressed
  if (warp == 8) tmem_dealloc2(tmem, 512);
}

bool tc_supported(int Ed, int Xd) { return (Ed == 64 && Xd == 16) || (Ed == 16 && Xd == 8); }

cudaError_t tc_layers_configure() {
  cudaError_t e = cudaFuncSetAttribute(k_layers_tc<64, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)LAYERS_SMEM_BYTES);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(k_layers_tc<16, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LAYERS_SMEM_BYTES);
}

void launch_layers_tc(cudaStream_t st, const Plan& p, const Dims& d, const EmbedW& ew, const LayerSched& q,
                      const Work& w, int num_sms) {
  int grid = 2 * q.nitems < num_sms ? 2 * q.nitems : num_sms;
  grid &= ~1;                                       // CTA pairs
  if (d.Ed == 64) k_layers_tc<64, 16><<<grid, LAYERS_THREADS, LAYERS_SMEM_BYTES, st>>>(p, d, ew, q, w);
  else k_layers_tc<16, 8><<<grid, LAYERS_THREADS, LAYERS_SMEM_BYTES, st>>>(p, d, ew, q, w);
}

}  // namespace bdiff
