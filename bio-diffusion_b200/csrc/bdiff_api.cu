// bdiff_api.cu — the C ABI declared in include/bdiff.h: handle, weight repacking, topology plan, forward,
// reverse step.  Host-side logic only; kernels live in bdiff_kernels_fp32.cu / bdiff_edge_tc.cu.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "../../include/bdiff.h"
#include "bdiff_handle.h"

using namespace bdiff;

namespace {

thread_local std::string g_create_error;


}  // namespace

namespace {

// ------------------------------------------------------------------------------------------ weight layout
void gcp_names(std::map<std::string, bool>& seen, const std::string& p, bool ff, bool vout) {
  seen[p + "vector_down.weight"] = false;
  seen[p + "vector_down_frames.weight"] = false;
  if (ff) {
    seen[p + "scalar_out.0.weight"] = false; seen[p + "scalar_out.0.bias"] = false;
    seen[p + "scalar_out.2.weight"] = false; seen[p + "scalar_out.2.bias"] = false;
  } else {
    seen[p + "scalar_out.weight"] = false; seen[p + "scalar_out.bias"] = false;
  }
  if (vout) {
    seen[p + "vector_up.weight"] = false;
    seen[p + "vector_out_scale.weight"] = false; seen[p + "vector_out_scale.bias"] = false;
  }
}

size_t layout_weights(bdiff_handle* h, bool assign) {
  // When !assign only the size is computed (wbuf is null); offsets are deterministic so a second pass assigns.
  const Dims& d = h->d;
  h->wused = 0;
  auto A = [&](size_t n) -> float* { float* r = h->walloc(n); return assign ? r : nullptr; };
  EmbedW& e = h->embed;
  e.eWs = A((size_t)d.Ke * d.Ed); e.ebs = A(d.Ed); e.ewd = A(d.Xd); e.ewf = A(4);
  e.eWu = A((size_t)d.Xd * d.Xd); e.eWg = A((size_t)d.Ed * d.Xd); e.ebg = A(d.Xd);
  e.nWs = A((size_t)d.Kn * 256); e.nbs = A(256); e.nWd = A(2 * 32); e.nWf = A(2 * 3 + 2);
  e.nWu = A(32 * 32); e.nWg = A(256 * 32); e.nbg = A(32);
  e.pWs = A((size_t)300 * d.Hin); e.pbs = A(d.Hin); e.pWd = A(32 * 32); e.pWf = A(32 * 3);
  h->layers.assign(d.L, LayerW{});
  for (int l = 0; l < d.L; ++l) {
    LayerW& w = h->layers[l];
    w.W0e = A((size_t)d.K0 * 256); w.Wsi = A(256 * 256); w.Wsj = A(256 * 256); w.b0 = A(256);
    w.Wd0i = A(32 * d.hid0); w.Wd0x = A((size_t)d.Xd * d.hid0); w.Wd0j = A(32 * d.hid0);
    w.Wf0i = A(32 * 3); w.Wf0x = A(d.Xd * 3); w.Wf0j = A(32 * 3);
    w.Wu0 = A(d.hid0 * 32); w.Wg0 = A(256 * 32); w.bg0 = A(32);
    for (int k = 0; k < 3; ++k) {
      w.Wk[k] = A((size_t)kKM * 256); w.bk[k] = A(256); w.Wdk[k] = A(32 * kHidM); w.Wfk[k] = A(32 * 3);
      w.Wuk[k] = A(kHidM * 32); w.Wgk[k] = A(256 * 32); w.bgk[k] = A(32);
    }
    w.wa = A(256); w.ba = A(4);
    w.W1 = A((size_t)kKFF * 256); w.b1 = A(256); w.W2 = A(256 * 256); w.b2 = A(256);
    w.Wdf = A(64 * kHidFF); w.Wff = A(64 * 3); w.Wuf = A(kHidFF * 32); w.Wgf = A(256 * 32); w.bgf = A(32);
    w.Wp = A((size_t)kKM * 256); w.bp = A(256); w.Wdp = A(32 * kHidM); w.Wfp = A(32 * 3);
    w.Wup = A(kHidM); w.Wgp = A(256); w.bgp = A(4);
  }
  return h->wused;
}

struct PackOp {
  const float* dst; int dst_ld; int col0; int ncols; int kpad; int nout;
};

// Resolve a reference parameter name to its pack operations + expected shape.
bool resolve(bdiff_handle* h, const std::string& name, std::vector<PackOp>& ops, int64_t& rows, int64_t& cols) {
  const Dims& d = h->d;
  auto W = [&](const float* dst, int dst_ld, int col0, int ncols, int kpad, int nout) {
    ops.push_back(PackOp{dst, dst_ld, col0, ncols, kpad, nout});
  };
  auto gcp = [&](const std::string& leaf, const float* Ws, int s_in, int kpad_s, int nout_s, const float* bs,
                 const float* Wd, int v_in, int hid, const float* Wf, const float* Wu, int v_out,
                 const float* Wg, const float* bg) -> bool {
    const int fan = s_in + hid + 9;
    if (leaf == "scalar_out.weight") { rows = nout_s; cols = fan; W(Ws, nout_s, 0, fan, kpad_s, nout_s); return true; }
    if (leaf == "scalar_out.bias") { rows = nout_s; cols = 1; W(bs, nout_s, 0, 1, 1, nout_s); return true; }
    if (leaf == "vector_down.weight") { rows = hid; cols = v_in; W(Wd, hid, 0, v_in, v_in, hid); return true; }
    if (leaf == "vector_down_frames.weight") { rows = 3; cols = v_in; W(Wf, 3, 0, v_in, v_in, 3); return true; }
    if (Wu && leaf == "vector_up.weight") { rows = v_out; cols = hid; W(Wu, v_out, 0, hid, hid, v_out); return true; }
    if (Wg && leaf == "vector_out_scale.weight") { rows = v_out; cols = nout_s; W(Wg, v_out, 0, nout_s, nout_s, v_out); return true; }
    if (bg && leaf == "vector_out_scale.bias") { rows = v_out; cols = 1; W(bg, v_out, 0, 1, 1, v_out); return true; }
    return false;
  };
  const EmbedW& e = h->embed;
  const std::string pe = "gcp_embedding.edge_embedding.", pn = "gcp_embedding.node_embedding.",
                    pp = "scalar_node_projection_gcp.";
  if (name.rfind(pe, 0) == 0)
    return gcp(name.substr(pe.size()), e.eWs, 1, d.Ke, d.Ed, e.ebs, e.ewd, 1, d.Xd, e.ewf, e.eWu, d.Xd, e.eWg, e.ebg);
  if (name.rfind(pn, 0) == 0)
    return gcp(name.substr(pn.size()), e.nWs, d.Hin, d.Kn, 256, e.nbs, e.nWd, 2, 32, e.nWf, e.nWu, 32, e.nWg, e.nbg);
  if (name.rfind(pp, 0) == 0)
    return gcp(name.substr(pp.size()), e.pWs, 256, 300, d.Hin, e.pbs, e.pWd, 32, 32, e.pWf, nullptr, 0, nullptr, nullptr);
  int l = -1, consumed = 0;
  if (sscanf(name.c_str(), "interaction_layers.%d.%n", &l, &consumed) != 1 || l < 0 || l >= d.L) return false;
  const std::string rest = name.substr(consumed);
  const LayerW& w = h->layers[l];
  const std::string pm = "interaction.message_fusion.", pa = "interaction.scalar_message_attention.0.",
                    pf = "feedforward_network.0.", px = "node_position_update_gcp.";
  if (rest.rfind(pm, 0) == 0) {
    int k = -1, c2 = 0;
    if (sscanf(rest.c_str() + pm.size(), "%d.%n", &k, &c2) != 1 || k < 0 || k > 3) return false;
    const std::string leaf = rest.substr(pm.size() + c2);
    if (k > 0)
      return gcp(leaf, w.Wk[k - 1], 256, kKM, 256, w.bk[k - 1], w.Wdk[k - 1], 32, kHidM, w.Wfk[k - 1], w.Wuk[k - 1],
                 32, w.Wgk[k - 1], w.bgk[k - 1]);
    // k == 0: split form.  Torch columns of scalar_out: [h_row(256) | e(Ed) | h_col(256) | vn(hid0) | q(9)],
    // of vector_down / vector_down_frames: [chi_row(32) | xi(Xd) | chi_col(32)]   (gcpnet.py:694)
    const int fan = 512 + d.Ed + d.hid0 + 9, vin = 64 + d.Xd;
    if (leaf == "scalar_out.weight") {
      rows = 256; cols = fan;
      W(w.Wsi, 256, 0, 256, 256, 256);
      W(w.Wsj, 256, 256 + d.Ed, 256, 256, 256);
      W(w.W0e, 256, 256, d.Ed, d.Ed, 256);                                             // e rows
      W(w.W0e + (size_t)d.Ed * 256, 256, 512 + d.Ed, d.hid0 + 9, d.K0 - d.Ed, 256);     // vn, q rows + zero pad
      return true;
    }
    if (leaf == "scalar_out.bias") { rows = 256; cols = 1; W(w.b0, 256, 0, 1, 1, 256); return true; }
    if (leaf == "vector_down.weight") {
      rows = d.hid0; cols = vin;
      W(w.Wd0i, d.hid0, 0, 32, 32, d.hid0); W(w.Wd0x, d.hid0, 32, d.Xd, d.Xd, d.hid0);
      W(w.Wd0j, d.hid0, 32 + d.Xd, 32, 32, d.hid0);
      return true;
    }
    if (leaf == "vector_down_frames.weight") {
      rows = 3; cols = vin;
      W(w.Wf0i, 3, 0, 32, 32, 3); W(w.Wf0x, 3, 32, d.Xd, d.Xd, 3); W(w.Wf0j, 3, 32 + d.Xd, 32, 32, 3);
      return true;
    }
    if (leaf == "vector_up.weight") { rows = 32; cols = d.hid0; W(w.Wu0, 32, 0, d.hid0, d.hid0, 32); return true; }
    if (leaf == "vector_out_scale.weight") { rows = 32; cols = 256; W(w.Wg0, 32, 0, 256, 256, 32); return true; }
    if (leaf == "vector_out_scale.bias") { rows = 32; cols = 1; W(w.bg0, 32, 0, 1, 1, 32); return true; }
    return false;
  }
  if (rest.rfind(pa, 0) == 0) {
    const std::string leaf = rest.substr(pa.size());
    if (leaf == "weight") { rows = 1; cols = 256; W(w.wa, 1, 0, 256, 256, 1); return true; }
    if (leaf == "bias") { rows = 1; cols = 1; W(w.ba, 1, 0, 1, 1, 1); return true; }
    return false;
  }
  if (rest.rfind(pf, 0) == 0) {
    const std::string leaf = rest.substr(pf.size());
    if (leaf == "scalar_out.0.weight") { rows = 256; cols = 537; W(w.W1, 256, 0, 537, kKFF, 256); return true; }
    if (leaf == "scalar_out.0.bias") { rows = 256; cols = 1; W(w.b1, 256, 0, 1, 1, 256); return true; }
    if (leaf == "scalar_out.2.weight") { rows = 256; cols = 256; W(w.W2, 256, 0, 256, 256, 256); return true; }
    if (leaf == "scalar_out.2.bias") { rows = 256; cols = 1; W(w.b2, 256, 0, 1, 1, 256); return true; }
    return gcp(leaf, nullptr, 512, 0, 256, nullptr, w.Wdf, 64, kHidFF, w.Wff, w.Wuf, 32, w.Wgf, w.bgf);
  }
  if (rest.rfind(px, 0) == 0)
    return gcp(rest.substr(px.size()), w.Wp, 256, kKM, 256, w.bp, w.Wdp, 32, kHidM, w.Wfp, w.Wup, 1, w.Wgp, w.bgp);
  return false;
}

cudaError_t ensure_work(bdiff_handle* h) {
  const Dims& d = h->d;
  const size_t Np = h->Npad, Ep = (size_t)h->Epad;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off += (n + 63) / 64 * 64; return o; };
  const size_t o_xi = take(Np * 3), o_x = take(Np * 3), o_hin = take(Np * d.Hin), o_chin = take(Np * 6),
               o_fbar = take(Np * 12), o_h = take(Np * 256), o_chi = take(Np * 96), o_PI = take(Np * kPStride),
               o_PJ = take(Np * kPStride), o_agg = take(Np * kMsg), o_hp = take(Np * 32),
               o_e = take(Ep * d.Ed), o_xie = take(Ep * d.Xd * 3), o_fr = take(Ep * 9), o_pjt = take(Np * 256),
               o_mid = take(h->cfg.mode == BDIFF_MODE_TENSOR ? (Ep / 128) * kMsg : 0),
               o_flag = take(64);
  cudaError_t e = h->work_buf.ensure(off * sizeof(float));
  if (e != cudaSuccess) return e;
  float* b = static_cast<float*>(h->work_buf.p);
  Work& w = h->work;
  w.x_init = b + o_xi; w.x = b + o_x; w.h_in = b + o_hin; w.chi_in = b + o_chin; w.fbar = b + o_fbar;
  w.h = b + o_h; w.chi = b + o_chi; w.PI = b + o_PI; w.PJ = b + o_PJ; w.agg = b + o_agg; w.hproj = b + o_hp;
  w.e = b + o_e; w.xi = b + o_xie; w.frames = b + o_fr;
  w.PJT = h->cfg.mode == BDIFF_MODE_TENSOR ? b + o_pjt : nullptr;
  w.mid = h->cfg.mode == BDIFF_MODE_TENSOR ? b + o_mid : nullptr;
  w.npad = (int)Np;
  w.nan_flag = reinterpret_cast<int*>(b + o_flag);
  w.dbg = nullptr;
  if (getenv("BDIFF_TIMING")) {
    e = h->dbg_buf.ensure(2 * 256 * 64 * sizeof(long long));
    if (e != cudaSuccess) return e;
    w.dbg = static_cast<long long*>(h->dbg_buf.p);
  }
  e = h->eps_buf.ensure(Np * (3 + d.F) * sizeof(float));
  if (e != cudaSuccess) return e;
  return h->tu_buf.ensure(256);
}

}  // namespace

extern "C" {

int32_t bdiff_abi_version(void) { return BDIFF_ABI_VERSION; }

int32_t bdiff_tc_edge_stream_layout(int32_t e_hidden, int32_t xi_hidden, int64_t* out) {
  if (!out || !tc_supported(e_hidden, xi_hidden)) return BDIFF_EINVAL;
  tc_edge_stream_layout(e_hidden, xi_hidden, out);
  return 0;
}

const char* bdiff_last_error(const bdiff_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int32_t bdiff_create(const bdiff_config* cfg, bdiff_handle** out) {
  if (!cfg || !out) { g_create_error = "null argument"; return BDIFF_EINVAL; }
  *out = nullptr;
  if (cfg->h_hidden != 256 || cfg->chi_hidden != 32) { g_create_error = "h_hidden must be 256 and chi_hidden 32"; return BDIFF_EINVAL; }
  if (cfg->e_hidden < 4 || cfg->e_hidden > 64 || cfg->e_hidden % 4) { g_create_error = "e_hidden must be a multiple of 4 in [4,64]"; return BDIFF_EINVAL; }
  if (cfg->xi_hidden < 4 || cfg->xi_hidden > 16 || cfg->xi_hidden % 4) { g_create_error = "xi_hidden must be a multiple of 4 in [4,16]"; return BDIFF_EINVAL; }
  if (cfg->num_h < 1 || cfg->num_context < 0 || cfg->num_h + 1 + cfg->num_context > 28) { g_create_error = "num_h + 1 + num_context must be in [2,28]"; return BDIFF_EINVAL; }
  if (cfg->num_layers < 1 || cfg->num_layers > 64) { g_create_error = "num_layers out of range"; return BDIFF_EINVAL; }
  if (cfg->mode != BDIFF_MODE_PARITY_FP32 && cfg->mode != BDIFF_MODE_TENSOR) { g_create_error = "unknown mode"; return BDIFF_EINVAL; }
  int dev_count = 0;
  if (cudaGetDeviceCount(&dev_count) != cudaSuccess || dev_count == 0) {
    g_create_error = "no CUDA device: libbdiff_sm100 has no CPU fallback";
    return BDIFF_ECUDA;
  }
  cudaDeviceProp prop{};
  int dev = 0;
  cudaGetDevice(&dev);
  cudaGetDeviceProperties(&prop, dev);
  if (prop.major != 10) {
    g_create_error = "libbdiff_sm100 is built for sm_100a (B200) only; found compute capability " +
                     std::to_string(prop.major) + "." + std::to_string(prop.minor);
    return BDIFF_ECUDA;
  }
  bdiff_handle* h = new bdiff_handle();
  h->cfg = *cfg;
  Dims& d = h->d;
  d.F = cfg->num_h; d.C = cfg->num_context; d.Hin = d.F + 1 + d.C; d.Ed = cfg->e_hidden; d.Xd = cfg->xi_hidden;
  d.hid0 = (64 + d.Xd) / 4;
  d.K0 = round_up(d.Ed + d.hid0 + 9, 4);
  d.Ke = round_up(1 + d.Xd + 9, 4);
  d.Kn = round_up(d.Hin + 32 + 9, 4);
  d.L = cfg->num_layers;
  if ((64 + d.Xd) % 4) { g_create_error = "2*chi_hidden + xi_hidden must be divisible by the bottleneck 4"; delete h; return BDIFF_EINVAL; }
  const size_t need = layout_weights(h, false);
  if (cudaMalloc(&h->wbuf, need * sizeof(float)) != cudaSuccess) { g_create_error = "cudaMalloc(weights) failed"; delete h; return BDIFF_ENOMEM; }
  cudaMemset(h->wbuf, 0, need * sizeof(float));
  h->wfloats = need;
  layout_weights(h, true);
  // the set of reference parameter names this configuration must receive
  gcp_names(h->seen, "gcp_embedding.edge_embedding.", false, true);
  gcp_names(h->seen, "gcp_embedding.node_embedding.", false, true);
  gcp_names(h->seen, "scalar_node_projection_gcp.", false, false);
  for (int l = 0; l < d.L; ++l) {
    const std::string p = "interaction_layers." + std::to_string(l) + ".";
    for (int k = 0; k < 4; ++k) gcp_names(h->seen, p + "interaction.message_fusion." + std::to_string(k) + ".", false, true);
    h->seen[p + "interaction.scalar_message_attention.0.weight"] = false;
    h->seen[p + "interaction.scalar_message_attention.0.bias"] = false;
    gcp_names(h->seen, p + "feedforward_network.0.", true, true);
    gcp_names(h->seen, p + "node_position_update_gcp.", false, true);
  }
  for (auto& kv : h->seen) {
    std::vector<PackOp> ops;
    int64_t rows = 0, cols = 0;
    if (!resolve(h, kv.first, ops, rows, cols)) { g_create_error = "internal: cannot place " + kv.first; cudaFree(h->wbuf); delete h; return BDIFF_EINVAL; }
    const size_t count = (size_t)rows * (size_t)cols;
    h->param_layout[kv.first] = {h->param_floats, count};
    h->param_floats += (count + 63) / 64 * 64;
  }
  h->num_sms = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    h->side = nullptr;               // fall back to a single stream
  }
  cudaError_t e = configure_kernels();
  if (e == cudaSuccess && cfg->mode == BDIFF_MODE_TENSOR) {
    if (!tc_supported(d.Ed, d.Xd)) {
      g_create_error = "tensor mode supports (e_hidden, xi_hidden) in {(64,16), (16,8)} only";
      cudaFree(h->wbuf);
      delete h;
      return BDIFF_EINVAL;
    }
    e = tc_layers_configure();
    h->tc_layer_bytes = tc_blob_bytes(d.Ed, d.Xd);
    h->tc_node_layer_bytes = tc_node_blob_bytes();
    if (e == cudaSuccess) e = h->tc_blob.ensure(h->tc_layer_bytes * d.L);
    if (e == cudaSuccess) e = h->tc_node_blob.ensure(h->tc_node_layer_bytes * d.L);
  }
  if (e != cudaSuccess) {
    g_create_error = std::string("configure_kernels: ") + cudaGetErrorString(e);
    cudaFree(h->wbuf);
    delete h;
    return BDIFF_ECUDA;
  }
  *out = h;
  return BDIFF_OK;
}

void bdiff_destroy(bdiff_handle* h) {
  if (!h) return;
  if (h->wbuf) cudaFree(h->wbuf);
  if (h->train) train_destroy(h->train);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->side) cudaStreamDestroy(h->side);
  h->plan_buf.release(); h->rc_buf.release(); h->layers_dev.release(); h->sched_buf.release(); h->items_buf.release(); h->work_buf.release(); h->eps_buf.release(); h->tu_buf.release(); h->tc_blob.release(); h->tc_node_blob.release(); h->stage_buf.release(); h->jobs_dev.release();
  delete h;
}

int32_t bdiff_set_weight(bdiff_handle* h, void* stream, const char* name, const float* data, const int64_t* shape,
                         int32_t ndim) {
  if (!h || !name || !data || !shape || ndim < 1 || ndim > 2) return h ? h->fail(BDIFF_EINVAL, "bad argument") : BDIFF_EINVAL;
  auto it = h->seen.find(name);
  if (it == h->seen.end()) return h->fail(BDIFF_EINVAL, "unknown parameter name '%s'", name);
  std::vector<PackOp> ops;
  int64_t rows = 0, cols = 0;
  if (!resolve(h, name, ops, rows, cols)) return h->fail(BDIFF_EINVAL, "cannot place parameter '%s'", name);
  const int64_t got_rows = shape[0], got_cols = ndim == 2 ? shape[1] : 1;
  if (got_rows != rows || got_cols != cols)
    return h->fail(BDIFF_EINVAL, "parameter '%s': expected shape [%lld,%lld], got [%lld,%lld]", name, (long long)rows,
                   (long long)cols, (long long)got_rows, (long long)got_cols);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // raw copy into the staging area (device-to-device, stream ordered); the repack of all slices is one kernel in bdiff_prepare
  const size_t count = (size_t)rows * (size_t)cols;
  cudaError_t e = h->stage_buf.p ? cudaSuccess : h->stage_buf.ensure((h->wfloats + 64 * h->seen.size()) * sizeof(float));
  if (e != cudaSuccess) return h->fail(BDIFF_ENOMEM, "weight staging: %s", cudaGetErrorString(e));
  auto so = h->stage_off.find(name);
  size_t off;
  if (so == h->stage_off.end()) {
    off = h->stage_used;
    h->stage_used += (count + 63) / 64 * 64;
    if (h->stage_used * sizeof(float) > h->stage_buf.bytes) return h->fail(BDIFF_ENOMEM, "weight staging overflow");
    h->stage_off[name] = off;
    const float* src = static_cast<const float*>(h->stage_buf.p) + off;
    for (const PackOp& op : ops) {
      PackJob j{const_cast<float*>(op.dst), src, op.dst_ld, (int)cols, op.col0, op.ncols, op.kpad, op.nout, h->pack_blocks};
      h->pack_blocks += (op.kpad * op.nout + 255) / 256;
      h->jobs.push_back(j);
    }
    h->jobs_uploaded = false;
  } else {
    off = so->second;
  }
  e = cudaMemcpyAsync(static_cast<float*>(h->stage_buf.p) + off, data, count * sizeof(float), cudaMemcpyDeviceToDevice, st);
  if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "stage '%s': %s", name, cudaGetErrorString(e));
  it->second = true;
  h->pack_dirty = true;
  h->tc_dirty = true;
  return BDIFF_OK;
}

static void tc_prepare(bdiff_handle* h, cudaStream_t st) {
  if (h->pack_dirty) {
    if (!h->jobs_uploaded && h->jobs_dev.ensure(h->jobs.size() * sizeof(PackJob)) == cudaSuccess) {
      cudaMemcpyAsync(h->jobs_dev.p, h->jobs.data(), h->jobs.size() * sizeof(PackJob), cudaMemcpyHostToDevice, st);
      cudaStreamSynchronize(st);    // pageable source; once per slice-table change, never inside a graph capture
      h->jobs_uploaded = true;
    }
    launch_pack_multi(st, static_cast<const PackJob*>(h->jobs_dev.p), (int)h->jobs.size(), h->pack_blocks);
    h->launches++;
    h->pack_dirty = false;
  }
  if (h->cfg.mode != BDIFF_MODE_TENSOR || !h->tc_dirty) return;
  for (int l = 0; l < h->d.L; ++l) {
    launch_tc_pack(st, h->layers[l], h->d, static_cast<unsigned char*>(h->tc_blob.p) + (size_t)l * h->tc_layer_bytes);
    const int last = (l == h->d.L - 1);
    unsigned char* nb = static_cast<unsigned char*>(h->tc_node_blob.p) + (size_t)l * h->tc_node_layer_bytes;
    launch_tc_pack_node(st, h->layers[l], h->layers[last ? l : l + 1], h->embed, h->d, last, nb);
    h->launches += 2;
  }
  if (h->layers_dev.ensure(h->layers.size() * sizeof(LayerW)) == cudaSuccess) {
    cudaMemcpyAsync(h->layers_dev.p, h->layers.data(), h->layers.size() * sizeof(LayerW), cudaMemcpyHostToDevice, st);
    cudaStreamSynchronize(st);      // pageable source; runs once per weight update, never inside a graph capture
  }
  h->tc_dirty = false;
}

int32_t bdiff_prepare(bdiff_handle* h, void* stream) {
  if (!h) return BDIFF_EINVAL;
  if (bdiff_weights_missing(h) != 0) return h->fail(BDIFF_ESTATE, "%d parameters not set", bdiff_weights_missing(h));
  tc_prepare(h, static_cast<cudaStream_t>(stream));
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? BDIFF_OK : h->fail(BDIFF_ECUDA, "prepare: %s", cudaGetErrorString(e));
}

int32_t bdiff_selftest_split(void* stream, int32_t variant, const float* A, const float* W, float* C) {
  if (!A || !W || !C) return BDIFF_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (selftest_configure() != cudaSuccess) return BDIFF_ECUDA;
  void* img = nullptr;
  if (cudaMalloc(&img, selftest_img_bytes()) != cudaSuccess) return BDIFF_ENOMEM;
  launch_umma_selftest_split(st, A, W, static_cast<unsigned char*>(img), C, variant);
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(img);
  return e == cudaSuccess ? BDIFF_OK : BDIFF_ECUDA;
}

int32_t bdiff_selftest_pair(void* stream, const float* A, const float* W, float* C) {
  if (!A || !W || !C) return BDIFF_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (selftest_pair_configure() != cudaSuccess) return BDIFF_ECUDA;
  void* img = nullptr;
  if (cudaMalloc(&img, selftest_pair_img_bytes()) != cudaSuccess) return BDIFF_ENOMEM;
  launch_umma_selftest_pair(st, A, W, static_cast<unsigned char*>(img), C);
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(img);
  return e == cudaSuccess ? BDIFF_OK : BDIFF_ECUDA;
}

int32_t bdiff_weights_missing(const bdiff_handle* h) {
  if (!h) return BDIFF_EINVAL;
  int n = 0;
  for (auto& kv : h->seen) n += kv.second ? 0 : 1;
  return n;
}

int32_t bdiff_plan_topology(bdiff_handle* h, void* stream, int32_t num_mols, int64_t num_nodes,
                            const int64_t* batch_index, const uint8_t* mask, int64_t* num_edges_host) {
  if (!h) return BDIFF_EINVAL;
  if (num_mols < 1 || num_nodes < 1 || !batch_index || !mask) return h->fail(BDIFF_EINVAL, "bad plan arguments");
  if (num_nodes > (1ll << 30)) return h->fail(BDIFF_EINVAL, "too many nodes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int N = (int)num_nodes, B = num_mols;
  std::vector<int64_t> bi(N);
  std::vector<uint8_t> mk(N);
  cudaError_t e = cudaMemcpyAsync(bi.data(), batch_index, N * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(mk.data(), mask, N, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "plan D2H: %s", cudaGetErrorString(e));
  std::vector<int> mol_off(B + 1, 0), act_off(B + 1, 0), act_idx, node_mol(N);
  std::vector<long long> edge_off(B + 1, 0);
  act_idx.reserve(N);
  int64_t prev = 0;
  for (int i = 0; i < N; ++i) {
    const int64_t m = bi[i];
    if (m < 0 || m >= B) return h->fail(BDIFF_EINVAL, "batch_index[%d]=%lld outside [0,%d)", i, (long long)m, B);
    if (m < prev) return h->fail(BDIFF_EINVAL, "batch_index must be sorted (node %d)", i);
    prev = m;
    mol_off[m + 1]++;
    node_mol[i] = (int)m;
  }
  for (int k = 0; k < B; ++k) mol_off[k + 1] += mol_off[k];
  for (int k = 0; k < B; ++k) {
    for (int i = mol_off[k]; i < mol_off[k + 1]; ++i)
      if (mk[i]) act_idx.push_back(i);
    act_off[k + 1] = (int)act_idx.size();
    const long long na = act_off[k + 1] - act_off[k];
    edge_off[k + 1] = edge_off[k] + na * na;
  }
  const long long E = edge_off[B];
  if (E >= (1ll << 36)) return h->fail(BDIFF_EINVAL, "too many edges");
  const size_t M = act_idx.size();
  // device layout: [mol_off | act_off | act_idx | node_mol | edge_off(int64) | mask]
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const long long ntile128 = (E + 127) / 128;
  std::vector<int> tile_mol((size_t)ntile128 + 1, 0);
  {
    int k = 0;
    for (long long t = 0; t < ntile128; ++t) {
      const long long g = t * 128;
      while (k < B && edge_off[k + 1] <= g) ++k;
      tile_mol[(size_t)t] = k;
    }
  }
  // dependency tables of the layer megakernel: edge tile -> 32-node tiles of its molecules, node tile -> edge tiles
  const int ntile32 = (N + 31) / 32;
  std::vector<int> edge_dep((size_t)2 * (ntile128 + 1), 0), node_dep((size_t)2 * (ntile32 + 1), 0);
  for (long long t = 0; t < ntile128; ++t) {
    const long long g1 = std::min<long long>(E, t * 128 + 128) - 1;
    int k0 = tile_mol[(size_t)t], k1 = k0;
    while (k1 < B - 1 && edge_off[k1 + 1] <= g1) ++k1;
    edge_dep[2 * t] = mol_off[k0] / 32;
    edge_dep[2 * t + 1] = (mol_off[k1 + 1] - 1) / 32;
  }
  for (int u = 0; u < ntile32; ++u) {
    const int n1 = std::min(N, u * 32 + 32) - 1;
    const int k0 = node_mol[u * 32], k1 = node_mol[n1];
    const long long e0 = edge_off[k0], e1 = edge_off[k1 + 1] - 1;
    node_dep[2 * u] = e1 >= e0 ? (int)(e0 / 128) : 0;
    node_dep[2 * u + 1] = e1 >= e0 ? (int)(e1 / 128) : -1;
  }
  // per node: edge tiles strictly inside its row (their sums go through Work::mid, see edge_tile_epilogue.inc)
  const int Npad128 = round_up(N, 128) + 128;          // node buffers carry one spare 128-row block (ghost node tile of an odd pair)
  std::vector<int> node_mid((size_t)2 * Npad128, 0);
  for (int k = 0; k < B; ++k) {
    const long long na = act_off[k + 1] - act_off[k];
    for (long long a = 0; a < na; ++a) {
      const long long g0 = edge_off[k] + a * na, g1 = g0 + na - 1;
      const long long t0 = g0 / 128, t1 = g1 / 128;
      if (t1 - t0 >= 2) {
        const int i = act_idx[act_off[k] + a];
        node_mid[2 * (size_t)i] = (int)(t0 + 1);
        node_mid[2 * (size_t)i + 1] = (int)(t1 - t0 - 1);
      }
    }
  }
  const size_t o_mo = take((B + 1) * 4), o_ao = take((B + 1) * 4), o_ai = take((M + 1) * 4), o_nm = take(N * 4),
               o_eo = take((B + 1) * 8), o_tm = take((ntile128 + 1) * 4), o_mk = take(N),
               o_ed = take((ntile128 + 1) * 8), o_nd = take((ntile32 + 1) * 8), o_mid = take((size_t)Npad128 * 8);
  std::vector<unsigned char> stage(off, 0);
  memcpy(stage.data() + o_mo, mol_off.data(), (B + 1) * 4);
  memcpy(stage.data() + o_ao, act_off.data(), (B + 1) * 4);
  if (M) memcpy(stage.data() + o_ai, act_idx.data(), M * 4);
  memcpy(stage.data() + o_nm, node_mol.data(), N * 4);
  memcpy(stage.data() + o_eo, edge_off.data(), (B + 1) * 8);
  memcpy(stage.data() + o_tm, tile_mol.data(), (size_t)(ntile128 + 1) * 4);
  memcpy(stage.data() + o_mk, mk.data(), N);
  memcpy(stage.data() + o_ed, edge_dep.data(), edge_dep.size() * 4);
  memcpy(stage.data() + o_nd, node_dep.data(), node_dep.size() * 4);
  memcpy(stage.data() + o_mid, node_mid.data(), node_mid.size() * 4);
  e = h->plan_buf.ensure(off);
  if (e == cudaSuccess) e = cudaMemcpyAsync(h->plan_buf.p, stage.data(), off, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "plan H2D: %s", cudaGetErrorString(e));
  unsigned char* base = static_cast<unsigned char*>(h->plan_buf.p);
  Plan& p = h->plan;
  p.B = B; p.N = N; p.E = E;
  p.mol_off = reinterpret_cast<int*>(base + o_mo);
  p.act_off = reinterpret_cast<int*>(base + o_ao);
  p.act_idx = reinterpret_cast<int*>(base + o_ai);
  p.node_mol = reinterpret_cast<int*>(base + o_nm);
  p.edge_off = reinterpret_cast<long long*>(base + o_eo);
  p.tile_mol = reinterpret_cast<int*>(base + o_tm);
  p.mask = base + o_mk;
  p.edge_rc = nullptr;
  p.node_mid = reinterpret_cast<const int2*>(base + o_mid);
  {
    const long long nrc = (ntile128 + 1) * 128;       // + one ghost tile (row = -1): the second CTA of the last pair when the tile count is odd
    e = h->rc_buf.ensure((size_t)(nrc > 0 ? nrc : 1) * sizeof(int4));
    if (e != cudaSuccess) return h->fail(BDIFF_ENOMEM, "plan edge records: %s", cudaGetErrorString(e));
    launch_edge_rc(st, p, static_cast<int4*>(h->rc_buf.p), nrc);
    p.edge_rc = static_cast<const int4*>(h->rc_buf.p);
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "plan edge records: %s", cudaGetErrorString(e));
  }
  h->sched.edge_dep = reinterpret_cast<const int2*>(base + o_ed);
  h->sched.node_dep = reinterpret_cast<const int2*>(base + o_nd);
  h->sched.TE = (int)ntile128;
  h->sched.TN = ntile32;
  {
    // Claim order of the layer megakernel, in PAIR items: a CTA pair works on tiles (2j, 2j+1) of one kind and layer (the
    // second tile of the last pair is a ghost when the count is odd).  Virtual time of edge pair (l, j) = l*PE + j; node pair
    // (l, v) follows the last edge pair it reads by `lag` claims (about one wave: by then that pair has normally finished).
    // Every dependency must precede its consumer in the list (deadlock freedom), which bounds the lag: edge pair (l+1, j)
    // reads node pairs <= ndep(j), whose time is l*PE + edep(ndep) + lag  <  (l+1)*PE + j.
    const int L = h->d.L, TE = (int)ntile128, TN = ntile32;
    const int PE = (TE + 1) / 2, PN = (TN + 1) / 2;
    if (L > 63 || ntile128 >= (1 << 24) || ntile32 >= (1 << 24)) return h->fail(BDIFF_EINVAL, "problem too large for the tile scheduler");
    auto node_pair_last_edge_pair = [&](int v) {          // last edge pair a node pair depends on (-1: none)
      int th = -1;
      for (int u = 2 * v; u < std::min(TN, 2 * v + 2); ++u) th = std::max(th, node_dep[2 * u + 1]);
      return th >= 0 ? th / 2 : -1;
    };
    auto edge_pair_last_node_pair = [&](int j) {
      int uh = -1;
      for (int t = 2 * j; t < std::min(TE, 2 * j + 2); ++t) uh = std::max(uh, edge_dep[2 * t + 1]);
      return uh >= 0 ? uh / 2 : -1;
    };
    long long lag = std::max(1, h->num_sms / 2);
    for (int j = 0; j < PE; ++j) {
      const int vh = edge_pair_last_node_pair(j);
      const int jh = (vh >= 0 && vh < PN) ? node_pair_last_edge_pair(vh) : -1;
      if (jh >= 0) lag = std::min<long long>(lag, (long long)PE - 1 - (jh - j));
    }
    if (lag < 0) lag = 0;
    std::vector<std::pair<long long, int>> order;
    order.reserve((size_t)L * (PE + PN));
    for (int l = 0; l < L; ++l) {
      for (int j = 0; j < PE; ++j) order.emplace_back(2 * ((long long)l * PE + j), (0 << 30) | (l << 24) | j);
      for (int v = 0; v < PN; ++v) {
        const int jh = node_pair_last_edge_pair(v);     // -1: no edges at all -> right at the start of the layer
        const long long tau = (long long)l * PE + (jh >= 0 ? jh + lag : 0);
        order.emplace_back(2 * tau + 1, (1 << 30) | (l << 24) | v);
      }
    }
    std::stable_sort(order.begin(), order.end(), [](const std::pair<long long, int>& a, const std::pair<long long, int>& b) { return a.first < b.first; });
    std::vector<int> items(order.size());
    for (size_t i = 0; i < order.size(); ++i) items[i] = order[i].second;
    e = h->items_buf.ensure(std::max<size_t>(items.size(), 1) * sizeof(int));
    if (e == cudaSuccess && !items.empty())
      e = cudaMemcpy(h->items_buf.p, items.data(), items.size() * sizeof(int), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return h->fail(BDIFF_ENOMEM, "scheduler work list: %s", cudaGetErrorString(e));
    h->sched.nitems = (int)items.size();
    h->sched.items = static_cast<const int*>(h->items_buf.p);
  }
  {
    const size_t nsched = 2 + (size_t)h->d.L * (size_t)(ntile128 + ntile32);
    e = h->sched_buf.ensure((nsched + 1) * sizeof(int));
    if (e != cudaSuccess) return h->fail(BDIFF_ENOMEM, "scheduler buffer: %s", cudaGetErrorString(e));
    h->sched.sched = static_cast<int*>(h->sched_buf.p);
    h->sched.err = h->sched.sched + nsched;
    cudaMemset(h->sched.err, 0, sizeof(int));
  }
  h->Npad = round_up(N, 128) + 128;
  h->Epad = (E + 127) / 128 * 128 + 128;
  e = ensure_work(h);
  if (e != cudaSuccess) return h->fail(BDIFF_ENOMEM, "workspace: %s", cudaGetErrorString(e));
  h->have_plan = true;
  h->plan_epoch++;
  h->Mact = (int)M;
  if (num_edges_host) *num_edges_host = E;
  return BDIFF_OK;
}

int32_t bdiff_edge_index(bdiff_handle* h, void* stream, int64_t* edge_index) {
  if (!h || !edge_index) return BDIFF_EINVAL;
  if (!h->have_plan) return h->fail(BDIFF_ESTATE, "no topology plan");
  launch_edge_index(static_cast<cudaStream_t>(stream), h->plan, reinterpret_cast<long long*>(edge_index));
  h->launches++;
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? BDIFF_OK : h->fail(BDIFF_ECUDA, "edge_index: %s", cudaGetErrorString(e));
}

static int32_t forward_impl(bdiff_handle* h, cudaStream_t st, const float* xh, const float* t_nodes,
                            const float* coef_table, const int* step_ptr, const float* context, float* net_out,
                            std::vector<cudaEvent_t>* ev = nullptr) {
  if (!h->have_plan) return h->fail(BDIFF_ESTATE, "bdiff_plan_topology has not been called");
  if (bdiff_weights_missing(h) != 0) {
    for (auto& kv : h->seen)
      if (!kv.second) return h->fail(BDIFF_ESTATE, "%d parameters not set, first missing: %s", bdiff_weights_missing(h), kv.first.c_str());
  }
  if (h->d.C > 0 && !context) return h->fail(BDIFF_EINVAL, "context required (num_context=%d)", h->d.C);
  const Plan& p = h->plan;
  const Dims& d = h->d;
  const Work& w = h->work;
  auto mark = [&]() {
    if (!ev) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    ev->push_back(e);
  };
  tc_prepare(h, st);
  const bool tensor = h->cfg.mode == BDIFF_MODE_TENSOR;
  mark();
  launch_prep(st, p, d, xh, t_nodes, coef_table, step_ptr, context, w);
  mark();
  // the edge embedding (e, xi, frames) and the node embedding (+ layer-0 endpoint projections) are independent and
  // neither fills the chip: run them side by side (fork/join through events; also valid under stream capture).
  // With per-kernel timing marks requested they stay in order on one stream.
  const bool fork = h->side != nullptr && ev == nullptr;
  if (fork) {
    cudaEventRecord(h->ev_fork, st);
    cudaStreamWaitEvent(h->side, h->ev_fork, 0);
    launch_edge_embed(h->side, p, d, h->embed, w);
    cudaEventRecord(h->ev_join, h->side);
  } else {
    launch_edge_embed(st, p, d, h->embed, w);
  }
  mark();
  launch_node_embed(st, p, d, h->embed, h->layers[0], w);
  if (fork) cudaStreamWaitEvent(st, h->ev_join, 0);
  mark();
  h->launches += 4;
  const bool fused = tensor;
  if (fused) {
    // all L layers in one persistent kernel (bdiff_layers_tc.cu); its queue head + completion flags are zeroed first
    LayerSched& q = h->sched;
    const size_t nsched = 2 + (size_t)d.L * (q.TE + q.TN);      // buffer sized in bdiff_plan_topology
    q.layers = static_cast<const LayerW*>(h->layers_dev.p);
    q.edge_blob = static_cast<const unsigned char*>(h->tc_blob.p);
    q.edge_blob_stride = h->tc_layer_bytes;
    q.node_blob = static_cast<const unsigned char*>(h->tc_node_blob.p);
    q.node_blob_stride = h->tc_node_layer_bytes;
    q.L = d.L;
    cudaMemsetAsync(q.sched, 0, nsched * sizeof(int), st);
    launch_layers_tc(st, p, d, h->embed, q, w, h->num_sms);
    mark();
    h->launches += 1;
  }
  for (int l = 0; l < d.L && !fused; ++l) {
    launch_edge_message(st, p, d, h->layers[l], w);
    mark();
    const bool last = (l == d.L - 1);
    launch_node_update(st, p, d, h->layers[l], h->layers[last ? l : l + 1], h->embed, w, last ? 1 : 0);
    mark();
    h->launches += 2;
  }
  launch_finalize(st, p, d, w, net_out);
  mark();
  h->launches += 1;
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? BDIFF_OK : h->fail(BDIFF_ECUDA, "forward: %s", cudaGetErrorString(e));
}

int32_t bdiff_profile_forward(bdiff_handle* h, void* stream, const float* xh, const float* t, const float* context,
                              float* net_out, float* ms_host) {
  if (!h || !xh || !t || !net_out || !ms_host) return h ? h->fail(BDIFF_EINVAL, "null argument") : BDIFF_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<cudaEvent_t> ev;
  int32_t rc = forward_impl(h, st, xh, t, nullptr, nullptr, context, net_out, &ev);
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc == BDIFF_OK && e != cudaSuccess) rc = h->fail(BDIFF_ECUDA, "profile sync: %s", cudaGetErrorString(e));
  if (rc == BDIFF_OK && h->cfg.mode == BDIFF_MODE_TENSOR && h->sched_buf.p) {
    int flag = 0;
    cudaMemcpy(&flag, h->sched.err, sizeof(int), cudaMemcpyDeviceToHost);
    if (flag) { cudaMemset(h->sched.err, 0, sizeof(int)); rc = h->fail(BDIFF_ECUDA, "layer megakernel: a tile dependency wait timed out"); }
  }
  for (int i = 0; i < 8; ++i) ms_host[i] = 0.f;
  if (rc == BDIFF_OK) {
    auto dt = [&](size_t a, size_t b) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[a], ev[b]); return ms; };
    const int L = h->d.L;
    ms_host[0] = dt(0, 1); ms_host[1] = dt(1, 2); ms_host[2] = dt(2, 3);
    if (ev.size() == 6) {          // fused layers: [prep | edge_embed | node_embed | k_layers_tc | finalize]
      ms_host[3] = dt(3, 4);       // reported in the edge_message slot; ms_host[7] < 0 marks the fusion
      ms_host[5] = dt(4, 5);
      ms_host[6] = dt(0, 5);
      ms_host[7] = -(float)L;
    } else {
      for (int l = 0; l < L; ++l) { ms_host[3] += dt(3 + 2 * l, 4 + 2 * l); ms_host[4] += dt(4 + 2 * l, 5 + 2 * l); }
      ms_host[5] = dt(3 + 2 * L, 4 + 2 * L);
      ms_host[6] = dt(0, 4 + 2 * L);
      ms_host[7] = (float)L;
    }
  }
  for (cudaEvent_t x : ev) cudaEventDestroy(x);
  return rc;
}

int32_t bdiff_denoise_forward(bdiff_handle* h, void* stream, const float* xh, const float* t, const float* context,
                              float* net_out) {
  if (!h || !xh || !t || !net_out) return h ? h->fail(BDIFF_EINVAL, "null argument") : BDIFF_EINVAL;
  return forward_impl(h, static_cast<cudaStream_t>(stream), xh, t, nullptr, nullptr, context, net_out);
}

int32_t bdiff_debug_tap(bdiff_handle* h, void* stream, const char* which, float* dst, int64_t* rows, int64_t* cols) {
  if (!h || !which || !rows || !cols) return BDIFF_EINVAL;
  if (!h->have_plan) return h->fail(BDIFF_ESTATE, "no topology plan");
  const std::string s = which;
  const Work& w = h->work;
  const Dims& d = h->d;
  const int64_t N = h->plan.N, E = h->plan.E;
  const float* src = nullptr;
  if (s == "f_ij") { src = w.frames; *rows = E; *cols = 9; }
  else if (s == "e") { src = w.e; *rows = E; *cols = d.Ed; }
  else if (s == "xi") { src = w.xi; *rows = E; *cols = d.Xd * 3; }
  else if (s == "h") { src = w.h; *rows = N; *cols = 256; }
  else if (s == "chi") { src = w.chi; *rows = N; *cols = 96; }
  else if (s == "x") { src = w.x; *rows = N; *cols = 3; }
  else if (s == "fbar") { src = w.fbar; *rows = N; *cols = 12; }
  else if (s == "chi_in") { src = w.chi_in; *rows = N; *cols = 6; }
  else if (s == "dbg" && w.dbg) { src = reinterpret_cast<const float*>(w.dbg); *rows = 512; *cols = 128; }
  else return h->fail(BDIFF_EINVAL, "unknown tap '%s'", which);
  if (dst && *rows * *cols > 0) {
    cudaError_t e = cudaMemcpyAsync(dst, src, (size_t)(*rows) * (*cols) * sizeof(float), cudaMemcpyDeviceToDevice,
                                    static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "tap copy: %s", cudaGetErrorString(e));
  }
  return BDIFF_OK;
}

int32_t bdiff_reverse_step(bdiff_handle* h, void* stream, float* z, const float* context, const float* noise_x,
                           const float* noise_h, const float* coef_table, const int32_t* step_index) {
  if (!h || !z || !noise_x || !noise_h || !coef_table) return h ? h->fail(BDIFF_EINVAL, "null argument") : BDIFF_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* eps = static_cast<float*>(h->eps_buf.p);
  int32_t rc = forward_impl(h, st, z, nullptr, coef_table, step_index, context, eps);
  if (rc != BDIFF_OK) return rc;
  launch_step(st, h->plan, h->d, 0, z, eps, noise_x, noise_h, coef_table, step_index, z);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? BDIFF_OK : h->fail(BDIFF_ECUDA, "reverse_step: %s", cudaGetErrorString(e));
}

int32_t bdiff_decode_z0(bdiff_handle* h, void* stream, const float* z0, const float* context, const float* noise_x,
                        const float* noise_h, const float* coef, float* xh) {
  if (!h || !z0 || !noise_x || !noise_h || !coef || !xh) return h ? h->fail(BDIFF_EINVAL, "null argument") : BDIFF_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* eps = static_cast<float*>(h->eps_buf.p);
  int32_t rc = forward_impl(h, st, z0, nullptr, coef, nullptr, context, eps);
  if (rc != BDIFF_OK) return rc;
  launch_step(st, h->plan, h->d, 1, z0, eps, noise_x, noise_h, coef, nullptr, xh);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? BDIFF_OK : h->fail(BDIFF_ECUDA, "decode_z0: %s", cudaGetErrorString(e));
}

int32_t bdiff_center_noise(bdiff_handle* h, void* stream, const float* noise_x, const float* noise_h, float* z) {
  if (!h || !noise_x || !noise_h || !z) return h ? h->fail(BDIFF_EINVAL, "null argument") : BDIFF_EINVAL;
  if (!h->have_plan) return h->fail(BDIFF_ESTATE, "no topology plan");
  launch_step(static_cast<cudaStream_t>(stream), h->plan, h->d, 2, nullptr, nullptr, noise_x, noise_h, nullptr, nullptr, z);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? BDIFF_OK : h->fail(BDIFF_ECUDA, "center_noise: %s", cudaGetErrorString(e));
}

int32_t bdiff_check(bdiff_handle* h, void* stream) {
  if (!h) return BDIFF_EINVAL;
  cudaError_t e = cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "check: %s", cudaGetErrorString(e));
  if (h->cfg.mode == BDIFF_MODE_TENSOR && h->sched_buf.p && h->have_plan) {
    int flag = 0;
    e = cudaMemcpy(&flag, h->sched.err, sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "check: %s", cudaGetErrorString(e));
    if (flag) { cudaMemset(h->sched.err, 0, sizeof(int)); return h->fail(BDIFF_ECUDA, "layer megakernel: a tile dependency wait timed out"); }
  }
  return BDIFF_OK;
}

int32_t bdiff_nan_guard_count(bdiff_handle* h, void* stream, int64_t* count_host, int32_t reset) {
  if (!h || !count_host) return h ? h->fail(BDIFF_EINVAL, "null argument") : BDIFF_EINVAL;
  *count_host = 0;
  if (!h->have_plan) return BDIFF_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int v = 0;
  cudaError_t e = cudaMemcpyAsync(&v, h->work.nan_flag + 1, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && reset) e = cudaMemsetAsync(h->work.nan_flag + 1, 0, sizeof(int), st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return h->fail(BDIFF_ECUDA, "nan_guard_count: %s", cudaGetErrorString(e));
  *count_host = v;
  return BDIFF_OK;
}

int64_t bdiff_launch_count(const bdiff_handle* h) { return h ? h->launches : 0; }

}  // extern "C"
