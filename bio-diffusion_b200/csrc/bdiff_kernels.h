// bdiff_kernels.h — host-visible launchers of the CUDA kernels (internal; the public surface is include/bdiff.h)
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "bdiff_common.cuh"

namespace bdiff {

// Per-forward workspace (device, fp32).  Node buffers are padded to a multiple of 16 rows, edge buffers to a
// multiple of 128 rows, and zero-initialised, so tile kernels never bounds-check their stores.
struct Work {
  float* x_init;   // [N,3]  masked input positions (un-centred)
  float* x;        // [N,3]  current (centred, then updated) positions
  float* h_in;     // [N,Hin]
  float* chi_in;   // [N,2,3]
  float* fbar;     // [N,12] mean frame of each node's row (9 used)
  float* h;        // [N,256]
  float* chi;      // [N,96]
  float* PI;       // [N,328] endpoint projections for the next edge pass (row side, bias folded in)
  float* PJ;       // [N,328] (col side)
  float* PJT;      // [Npad/32][256][32] scalar part of PJ, column-major inside blocks of 32 nodes (tensor mode: consecutive
                   //             edges of a tile have consecutive target nodes -> coalesced per-edge gather), else nullptr
  int npad;        // row count of the padded node buffers
  float* agg;      // [N,352] aggregated messages
  float* mid;      // [ceil(E/128),352] tensor mode: message sums of edge tiles that lie strictly inside one source node's row
  float* hproj;    // [N,32]  projected scalar outputs (Hin used)
  float* e;        // [E,Ed]
  float* xi;       // [E,Xd*3]
  float* frames;   // [E,9]
  int* nan_flag;   // [0] NaN seen in this forward (gcpnet.py:1214-1216 guard), [1] forwards in which the guard fired (cumulative)
  long long* dbg;  // optional [CTA][64] clock64 stamps of the tensor-core kernels (BDIFF_TIMING=1), else nullptr
};

cudaError_t configure_kernels();
size_t edge_smem_bytes();
size_t node_smem_bytes();

void launch_prep(cudaStream_t st, const Plan& p, const Dims& d, const float* xh, const float* t_nodes,
                 const float* coef_table, const int* step_ptr, const float* ctx, const Work& w);
void launch_edge_embed(cudaStream_t st, const Plan& p, const Dims& d, const EmbedW& ew, const Work& w);
void launch_node_embed(cudaStream_t st, const Plan& p, const Dims& d, const EmbedW& ew, const LayerW& l0,
                       const Work& w);
void launch_edge_message(cudaStream_t st, const Plan& p, const Dims& d, const LayerW& lw, const Work& w);
void launch_node_update(cudaStream_t st, const Plan& p, const Dims& d, const LayerW& lw, const LayerW& wn,
                        const EmbedW& ew, const Work& w, int last);
void launch_finalize(cudaStream_t st, const Plan& p, const Dims& d, const Work& w, float* out);
void launch_step(cudaStream_t st, const Plan& p, const Dims& d, int mode, const float* z, const float* eps,
                 const float* noise_x, const float* noise_h, const float* coef_table, const int* step_ptr,
                 float* out);
void launch_edge_index(cudaStream_t st, const Plan& p, long long* out);
void launch_edge_rc(cudaStream_t st, const Plan& p, int4* out, long long n);
// one slice of a reference parameter tensor -> kernel layout (see k_pack_multi)
struct PackJob {
  float* dst;
  const float* src;
  int dst_ld, src_ld, col0, ncols, kpad, nout;
  int block0;              // first block of this job in the multi-slice launch (256 threads per block)
};
void launch_pack_multi(cudaStream_t st, const PackJob* jobs_dev, int njobs, int total_blocks);

// tensor mode: per-layer split-bf16 weight streams (bdiff_tc_pack.cu)
bool tc_supported(int Ed, int Xd);
size_t tc_blob_bytes(int Ed, int Xd);
void tc_edge_stream_layout(int Ed, int Xd, int64_t* out);   // {stream bytes, chunks per CTA and tile, chunk bytes of both CTAs}
size_t tc_node_blob_bytes();
void launch_tc_pack(cudaStream_t st, const LayerW& lw, const Dims& d, unsigned char* blob);
void launch_tc_pack_node(cudaStream_t st, const LayerW& lw, const LayerW& wn, const EmbedW& ew, const Dims& d, int last,
                         unsigned char* blob);
// all layers in one persistent kernel (bdiff_layers_tc.cu)
struct LayerSched {
  const LayerW* layers;            // [L] device copy of the per-layer weight pointer tables
  const unsigned char* edge_blob;  // per-layer bf16 blobs of the edge / node passes
  size_t edge_blob_stride;
  const unsigned char* node_blob;
  size_t node_blob_stride;
  int L, TE, TN;                   // layers, 128-edge tiles, 32-node tiles
  int nitems;                      // pair items in the work list: L * (ceil(TE/2) + ceil(TN/2))
  int* sched;                      // [0] queue head, [1] unused, [2 + l*(TE+TN) + i] completion flags; zeroed per forward
  int* err;                        // sticky error word (dependency wait timed out); cleared when the plan is built / reported
  const int2* edge_dep;            // [TE] inclusive range of 32-node tiles whose previous-layer output an edge tile reads
  const int2* node_dep;            // [TN] inclusive range of edge tiles whose messages a node tile reads
  const int* items;                // [nitems] work list in claim order: type<<30 | layer<<24 | PAIR index: a CTA pair works on tiles 2j, 2j+1 (see bdiff_plan_topology)
};
cudaError_t tc_layers_configure();
void launch_layers_tc(cudaStream_t st, const Plan& p, const Dims& d, const EmbedW& ew, const LayerSched& q,
                      const Work& w, int num_sms);
cudaError_t selftest_configure();
cudaError_t selftest_pair_configure();
size_t selftest_pair_img_bytes();
void launch_umma_selftest_pair(cudaStream_t st, const float* A, const float* W, unsigned char* img_scratch, float* C);
size_t selftest_img_bytes();
void launch_umma_selftest_split(cudaStream_t st, const float* A, const float* W, unsigned char* img_scratch, float* C,
                                int variant);

}  // namespace bdiff
