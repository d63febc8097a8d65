// bdiff_tc_pack.cu — per-layer weight streams of the tensor path: split-bf16 K=16 slabs (bdiff_slab.cuh) in exactly the
// order the megakernel's TMA lane streams them.  Runs once per weight update (bdiff_prepare).
#include "bdiff_node_tc.cuh"

namespace bdiff {

size_t tc_blob_bytes(int Ed, int Xd) { return tc_edge_stream_bytes(Ed, Xd); }
size_t tc_node_blob_bytes() { return tc_node_stream_bytes(0); }      // the last layer's stream is shorter
void tc_edge_stream_layout(int Ed, int Xd, int64_t* out) {
  const int k0s = tc_k0_steps(Ed, Xd);
  out[0] = (int64_t)tc_edge_stream_bytes(Ed, Xd);
  out[1] = tc_edge_tile_chunks(k0s);
  out[2] = (int64_t)tc_edge_chunks_total_bytes(k0s);
}

// A layer's stream is [CTA 0's half | CTA 1's half] (the megakernel runs CTA pairs, cta_group::2: an N-row plane is split between
// the two shared memories, CTA c supplying rows [c N/2, (c+1) N/2) of every MMA's B operand).  Per CTA, in streaming order:
// Edge pass:  G0: K0S steps x 128 local rows (W0e rows [128 c, 128 c + 128), zero-padded to K0S*16 K rows)
//             for k = 1..3:  U pass: 16 steps x 32 local gate rows (CTA 0 -> U0, CTA 1 -> U1), 4 steps per TMA chunk,
//                            S pass: 16 steps x 128 local rows (W_k rows 128 c .. +128),
//                            2 steps x 128 local rows (W_k K rows 256..287)
//             G4: 16 steps x 16 local rows (Wg_3 rows [16 c, 16 c + 16))
//             (tc_edge_chunk_bytes lists the TMA chunks of this order)
// Gate rows: GCP kk = gi + 1 adds +Wg_{kk-1} m_{kk-1} to U[(kk-1) & 1] and starts U[kk & 1] = -Wg_kk m_{kk-1} (sign folded into
// the packed weights so that U0 | U1 is one N=64 accumulator range).
// one thread per (global plane row, k in [0,16)); writes the hi and the lo plane element
__global__ void k_pack_edge_slabs(LayerW lw, Dims d, unsigned char* __restrict__ blob, size_t half_bytes) {
  const int K0S = tc_k0_steps(d.Ed, d.Xd);
  const long long rows_g = 16 * 320 + 2 * 256;
  const long long total_rows = (long long)K0S * 256 + 3 * rows_g + 16 * 32;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total_rows * 16) return;
  long long row = idx >> 4;
  const int kk = (int)(idx & 15);
  size_t base = 0;            // offset inside a CTA's stream
  int NL, n, k, cta, local;
  float v;
  if (row < (long long)K0S * 256) {
    const int step = (int)(row / 256);
    n = (int)(row % 256); NL = 128; cta = n >> 7; local = n & 127; base = (size_t)step * 2 * 128 * 32; k = step * 16 + kk;
    v = k < d.K0 ? lw.W0e[(size_t)k * 256 + n] : 0.f;
  } else {
    row -= (long long)K0S * 256;
    base = (size_t)K0S * 2 * 128 * 32;
    const size_t bytes_g = (size_t)16 * 2 * 160 * 32 + 2 * 2 * 128 * 32;
    if (row < 3 * rows_g) {
      const int gi = (int)(row / rows_g);
      long long rr = row - gi * rows_g;
      base += gi * bytes_g;
      if (rr < 16 * 320) {
        // global row n of K step `step`: W_k rows 0..255 go to the S pass (planes of 128 local rows, after the 16 gate
        // planes), the 64 gate rows to the U pass (planes of 32 local rows, 4 K steps per chunk)
        const int step = (int)(rr / 320);
        n = (int)(rr % 320); k = step * 16 + kk;
        const float* wprev = gi == 0 ? lw.Wg0 : lw.Wgk[gi - 1];
        const float* wthis = lw.Wgk[gi];
        const bool odd = ((gi + 1) & 1) != 0;           // kk odd: U0 <- +prev, U1 <- -this;  kk even: U0 <- -this, U1 <- +prev
        if (n < 256) {
          v = lw.Wk[gi][(size_t)k * 256 + n]; cta = n >> 7; local = n & 127;
          NL = 128; base += (size_t)16 * 2 * 32 * 32 + (size_t)step * 2 * 128 * 32;
        } else {
          if (n < 288) { v = odd ? wprev[(size_t)k * 32 + (n - 256)] : -wthis[(size_t)k * 32 + (n - 256)]; cta = 0; local = n - 256; }
          else { v = odd ? -wthis[(size_t)k * 32 + (n - 288)] : wprev[(size_t)k * 32 + (n - 288)]; cta = 1; local = n - 288; }
          NL = 32; base += (size_t)step * 2 * 32 * 32;
        }
      } else {
        rr -= 16 * 320;
        const int step = (int)(rr / 256);
        n = (int)(rr % 256); NL = 128; cta = n >> 7; local = n & 127;
        base += (size_t)16 * 2 * 160 * 32 + (size_t)step * 2 * 128 * 32; k = 256 + step * 16 + kk;
        v = k < kKM ? lw.Wk[gi][(size_t)k * 256 + n] : 0.f;
      }
    } else {
      row -= 3 * rows_g;
      base += 3 * bytes_g;
      const int step = (int)(row / 32);
      n = (int)(row % 32); NL = 16; cta = n >> 4; local = n & 15; base += (size_t)step * 2 * 16 * 32; k = step * 16 + kk;
      v = lw.Wgk[2][(size_t)k * 32 + n];
    }
  }
  slab_store(blob + (size_t)cta * half_bytes + base, NL, local, kk, v);
}

// Node pass, per CTA (issue order):  G1a 16x128: W1[0:256]   | G1b 16x144: W1[256:512] + 16 rows of -Wg_ff | G1c 2x128: W1[512:544]
//                                    G2 16x128: W2           | G3a 16x144: Wp[0:256] + 16 rows of Wg_ff    |
//   not last: G4 16x128: next.Wsi | G3b 2x128: Wp[256:288] | G5 16x128: next.Wsj
//   last:     G3b 2x128           | Gp 19x16: projection scalar_out (K = 300 -> 304, Hin -> 32 rows, zero padded)
__global__ void k_pack_node_slabs(LayerW lw, LayerW wn, EmbedW ew, Dims d, int last, unsigned char* __restrict__ blob,
                                  size_t half_bytes) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long row = idx >> 4;
  const int kk = (int)(idx & 15);
  size_t base = 0;
  int NL = 0, n = 0, k = 0, cta = 0, local = 0;
  float v = 0.f;
  bool found = false;
  // segment walker: `steps` K steps of NN-row global planes; sets (n, k), the CTA's local row / plane height and base
  auto seg = [&](int steps, int NN) -> bool {
    if (found) return false;
    const long long rows = (long long)steps * NN;
    const int nl = NN == 256 ? 128 : (NN == 288 ? 144 : 16);
    if (row < rows) {
      const int step = (int)(row / NN);
      n = (int)(row % NN); NL = nl; base += (size_t)step * 2 * nl * 32; k = step * 16 + kk;
      if (NN == 288 && n >= 256) { cta = (n - 256) >> 4; local = 128 + ((n - 256) & 15); }
      else if (NN == 32) { cta = n >> 4; local = n & 15; }
      else { cta = n >> 7; local = n & 127; }
      found = true;
      return true;
    }
    row -= rows;
    base += (size_t)steps * 2 * nl * 32;
    return false;
  };
  if (seg(16, 256)) v = lw.W1[(size_t)k * 256 + n];
  else if (seg(16, 288)) v = n < 256 ? lw.W1[(size_t)(256 + k) * 256 + n] : -lw.Wgf[(size_t)k * 32 + (n - 256)];   // U = -Wg h_old
  else if (seg(2, 256)) v = 512 + k < kKFF ? lw.W1[(size_t)(512 + k) * 256 + n] : 0.f;
  else if (seg(16, 256)) v = lw.W2[(size_t)k * 256 + n];
  else if (seg(16, 288)) v = n < 256 ? lw.Wp[(size_t)k * 256 + n] : lw.Wgf[(size_t)k * 32 + (n - 256)];
  else if (!last) {
    if (seg(16, 256)) v = wn.Wsi[(size_t)k * 256 + n];
    else if (seg(2, 256)) v = 256 + k < kKM ? lw.Wp[(size_t)(256 + k) * 256 + n] : 0.f;
    else if (seg(16, 256)) v = wn.Wsj[(size_t)k * 256 + n];
  } else {
    if (seg(2, 256)) v = 256 + k < kKM ? lw.Wp[(size_t)(256 + k) * 256 + n] : 0.f;
    else if (seg(19, 32)) v = (k < 300 && n < d.Hin) ? ew.pWs[(size_t)k * d.Hin + n] : 0.f;
  }
  if (!found) return;
  slab_store(blob + (size_t)cta * half_bytes + base, NL, local, kk, v);
}

void launch_tc_pack(cudaStream_t st, const LayerW& lw, const Dims& d, unsigned char* blob) {
  const long long rows = (long long)tc_k0_steps(d.Ed, d.Xd) * 256 + 3 * (16 * 320 + 2 * 256) + 16 * 32;
  const long long total = rows * 16;
  k_pack_edge_slabs<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(lw, d, blob, tc_blob_bytes(d.Ed, d.Xd) / 2);
}

void launch_tc_pack_node(cudaStream_t st, const LayerW& lw, const LayerW& wn, const EmbedW& ew, const Dims& d, int last,
                         unsigned char* blob) {
  const long long rows = 16 * 256 + 16 * 288 + 2 * 256 + 16 * 256 + 16 * 288 + (last ? 2 * 256 + 19 * 32 : 16 * 256 + 2 * 256 + 16 * 256);
  const long long total = rows * 16;
  k_pack_node_slabs<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(lw, wn, ew, d, last, blob, tc_node_blob_bytes() / 2);
}

}  // namespace bdiff
