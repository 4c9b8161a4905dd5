// engine.cu -- host orchestration behind the C-ABI (include/b200mlip.h):
// weight composition, GPU-resident workspace, forward + hand-derived backward schedule, halo exchange
// between slab neighbours (NCCL point-to-point between processes, peer-memory stores inside a
// single-process group), and the extern "C" entry points.
//
// Schedule mirrors (and is verified stage-by-stage against) oracle/manual_ref.py; the reference
// control flow it replaces is DistMLIP/implementations/matgl/models/chgnet.py:208-453 (forward)
// and pes.py:109-145 (scaling, autograd backward, forces, stress).
#include <dlfcn.h>
#include <nccl.h>

#include <cmath>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <cstring>
#include <map>
#include <new>
#include <set>
#include <string>
#include <vector>

#include <algorithm>

#include "graph.cuh"
#include "kernels.cuh"
#include "tn_state.cuh"

namespace b2m {

// ------------------------------------------------------------------------------------------
// NCCL through dlopen: if torch already loaded its bundled libnccl.so.2 we reuse that copy.
// ------------------------------------------------------------------------------------------
struct Nccl {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  void load() {
    if (lib) return;
    lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    B2M_REQUIRE(lib != nullptr, B2M_ERR_CUDA, "cannot dlopen libnccl.so.2 (needed for world > 1)");
#define L(name, sym)                                              \
  *(void**)(&name) = dlsym(lib, sym);                             \
  B2M_REQUIRE(name != nullptr, B2M_ERR_CUDA, "NCCL symbol missing: " sym)
    L(GetUniqueId, "ncclGetUniqueId");
    L(CommInitRank, "ncclCommInitRank");
    L(CommDestroy, "ncclCommDestroy");
    L(Send, "ncclSend");
    L(Recv, "ncclRecv");
    L(AllReduce, "ncclAllReduce");
    L(GroupStart, "ncclGroupStart");
    L(GroupEnd, "ncclGroupEnd");
    L(GetErrorString, "ncclGetErrorString");
#undef L
  }
};
static Nccl g_nccl;
#define NCCL_CK(call)                                                                              \
  do {                                                                                             \
    ncclResult_t r__ = (call);                                                                     \
    if (r__ != ncclSuccess)                                                                        \
      throw b2m::Error(B2M_ERR_CUDA, std::string("NCCL error: ") + g_nccl.GetErrorString(r__));   \
  } while (0)

// ------------------------------------------------------------------------------------------
struct AtomLayerW {
  float *W1s_k, *W1e_k, *W1t_k, *b1, *W1s_raw, *W1e_raw, *W1t_raw, *M, *W2k, *W2raw, *b2, *Wout_k, *Wout_raw;
  float *W2can, *Mcan, *W2Tcan;  // tcgen05 operands (canonical UMMA layout, tf32 hi/lo planes)
};
struct BondLayerW {
  float *W1a_k, *W1b_k, *W1c_k, *Wg_k, *b1, *W1a_raw, *W1b_raw, *W1c_raw, *Wg_raw, *W2k, *W2raw, *b2, *Wout_k, *Wout_raw;
  float *WAa_k, *WAb_k, *WAc_k, *WAg_k, *bA, *WAa_raw, *WAb_raw, *WAc_raw, *WAg_raw;
  float *Wgcan, *W2can, *W2Tcan, *WgTcan, *WAgcan, *WAgTcan;  // tcgen05 operands
};

}  // namespace b2m

using namespace b2m;

// Host-side rendezvous of the partition threads of a single-process group (b2m_create with ndev > 1).  abort() releases
// every waiter so that an exception in one partition cannot dead-lock the others.
struct GroupSync {
  std::mutex m;
  std::condition_variable cv;
  int n = 1, waiting = 0;
  long long gen = 0;
  bool aborted = false;
  void reset(int n_) { n = n_, waiting = 0, aborted = false; }
  void arrive_and_wait() {
    std::unique_lock<std::mutex> lk(m);
    if (aborted) throw b2m::Error(B2M_ERR_STATE, "a partition of the group failed");
    const long long my = gen;
    if (++waiting == n) {
      waiting = 0, gen++;
      cv.notify_all();
      return;
    }
    cv.wait(lk, [&] { return gen != my || aborted; });
    if (aborted && gen == my) throw b2m::Error(B2M_ERR_STATE, "a partition of the group failed");
  }
  void abort() {
    std::lock_guard<std::mutex> lk(m);
    aborted = true;
    cv.notify_all();
  }
};

struct b2m_engine {
  b2m_model_desc desc;
  int kind = 0;                   // 0: CHGNet (b2m_create), 1: TensorNet (b2m_create_tensornet)
  b2m::TnState* tn = nullptr;     // TensorNet weights and workspace (kind 1)
  int device = 0;
  cudaStream_t st = nullptr;
  cudaStream_t cst = nullptr;            // halo traffic of the forward pass (overlaps the projections that do not need it)
  cudaEvent_t ev_prod = nullptr, ev_halo = nullptr;
  std::string err;
  // weights
  std::map<std::string, std::vector<float>> host_w;
  std::map<std::string, std::vector<int64_t>> host_shape;
  std::set<std::string> consumed;  // state_dict keys finalize_weights actually used
  std::vector<double> elem_refs;
  DBuf<double> erefbuf;
  bool finalized = false;
  DBuf<float> wbuf;
  std::vector<AtomLayerW> aw;
  std::vector<BondLayerW> bw;
  float *d_emb = nullptr, *d_Wbe = nullptr, *d_Wae = nullptr, *d_Wabw = nullptr, *d_W3bw = nullptr, *d_fa = nullptr;
  float *d_F0k = nullptr, *d_c0 = nullptr, *d_F0raw = nullptr, *d_F1k = nullptr, *d_c1 = nullptr, *d_F1raw = nullptr,
        *d_F2 = nullptr, *d_Ws = nullptr;
  const double* d_eref = nullptr;  // per-element energy offsets, double like the energy accumulator
  float c2 = 0.f, bs = 0.f;
  RadialParams rp2, rp3;
  // comm
  int rank = 0, world = 1;
  ncclComm_t comm = nullptr;
  // single-process group (ndev > 1): the handle returned by b2m_create is parts[0]; every partition is a full engine on
  // its own device (ordinals may repeat) and stream, driven by its own host thread inside b2m_set_structure /
  // b2m_compute; halo rows travel as direct peer-memory stores / copies ordered by CUDA events (no NCCL)
  std::vector<b2m_engine*> parts;  // leader only: all partitions, parts[0] == this
  b2m_engine* leader = nullptr;    // members: the leader (for the peer table and the rendezvous)
  GroupSync gsync;                 // leader only
  std::vector<cudaEvent_t> hev;    // one event per halo-exchange point of a run
  int hpoint = 0;
  DBuf<float> precv[2];            // adjoint rows pushed by my neighbours (backward), double-buffered by point parity
  DBuf<float> ftmp;                // leader: staging of a peer's force array
  int view = 0;                    // leader: partition addressed by the inspection calls (b2m_set_view)
  // page-locked staging owned by the library: host arrays go through it with a few copy threads (a single-threaded
  // memcpy of 24 MB of positions was the largest host item of an end-to-end step at 1 M atoms)
  void* pin_in = nullptr;   // [N,3] f64 positions followed by [N] i32 species
  size_t pin_in_cap = 0;
  void* pin_out = nullptr;  // [N,3] f32 forces
  size_t pin_out_cap = 0;
  // graph + workspace
  Graph g;
  bool have_graph = false;
  std::vector<DBuf<float>> x, h, ang, upd, uv, uvB, dsB, uvA;
  DBuf<float> be_e, dbe_e;  // [E,12] radial basis and derivative, once per step
  bool want_grads = true;
  // per-atom output (b2m_compute_peratom): W_i rows [N][kAtomVirW] f32 and e_i [N] f64 in global order, allocated on the
  // first per-atom evaluation only; reduced over the partitions like `forces`
  bool want_peratom = false;
  DBuf<float> atom_vir, avtmp;  // avtmp / aetmp: leader's staging of a peer partition's arrays
  DBuf<double> atom_e, aetmp;
  // first-layer projections of every atom-conv layer (A = x W1s^T, C = x W1t^T + b1, Q = h W1e^T), one buffer per
  // layer: the backward gathers the rows the forward wrote instead of re-running three GEMMs per layer
  // (about 1.1 GB per 100k atoms for the four layers)
  std::vector<DBuf<float>> ApL, CpL, QpL;
  static int proj_slot(int l) { return l; }
  DBuf<float> Ha, Hb, Xc, agg, aggB, y1p, y1, y2p, y2, e_atom, site;
  DBuf<float> gx, gh, gang, gA, gC, gQ, gHa, gHb, gXc, gagg, gupd, gaggB, gd, gdb, gbvec, gy1, gy2;
  DBuf<float> forces, sendbuf, recvbuf, site_full;
  DBuf<double> scal;  // [0]=energy, [1..9]=virial
  // timings
  cudaEvent_t ev[8] = {nullptr};
  double t_graph = 0, t_fwd = 0, t_bwd = 0, t_gather = 0, t_total = 0;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> gather_ev;
  long long launches_last = 0;
  double last_energy = 0;
  std::map<const float*, const float*> canon_of;  // FFMA-layout GEMM operand -> canonical tcgen05 copy
  int num_sms = 148;
  bool use_tc = true;  // tcgen05 kernels; B2M_LEGACY_FFMA=1 selects the FP32-FFMA tile kernels (A/B checks)
  bool debug_no_halo = false;  // B2M_DEBUG_NO_HALO=1: a b2m_set_partition view may run with its exchanges skipped (wrong
                               // numbers, right amount of per-partition work: timing one slab of an N-way split on one GPU)
  int ac_gen = 3;      // atom-conv kernel generation on the tcgen05 path: 3 (default, kernels_ac3.cu), 1 = first generation,
                       // 4 = third-generation forward with the first-generation backward (B2M_ATOMCONV, A/B checks)
};

namespace b2m {

static const std::vector<float>& W(b2m_engine* e, const std::string& k, std::vector<int64_t> shape) {
  auto it = e->host_w.find(k);
  B2M_REQUIRE(it != e->host_w.end(), B2M_ERR_INVALID, "missing weight: " + k);
  e->consumed.insert(k);
  const auto& sh = e->host_shape[k];
  size_t n = 1;
  for (auto s : shape) n *= (size_t)s;
  B2M_REQUIRE(it->second.size() == n && sh == shape, B2M_ERR_INVALID,
              "weight '" + k + "' has an unsupported shape (engine supports dim=64, max_n=9, max_f=4)");
  return it->second;
}

struct Packer {
  std::vector<float> host;
  size_t add(const std::vector<float>& v) {
    size_t off = (host.size() + 63) / 64 * 64;  // 256 B alignment
    host.resize(off + v.size());
    memcpy(host.data() + off, v.data(), v.size() * sizeof(float));
    return off;
  }
};

// slice columns [c0, c0+64) of a row-major [rows][ncol] matrix -> [rows][64]
static std::vector<float> cols(const std::vector<float>& m, int rows, int ncol, int c0) {
  std::vector<float> o((size_t)rows * 64);
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < 64; c++) o[(size_t)r * 64 + c] = m[(size_t)r * ncol + c0 + c];
  return o;
}
static std::vector<float> transpose(const std::vector<float>& m, int rows, int ncol) {
  std::vector<float> o(m.size());
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < ncol; c++) o[(size_t)c * rows + r] = m[(size_t)r * ncol + c];
  return o;
}
static std::vector<float> vcat(const std::vector<float>& a, const std::vector<float>& b) {
  std::vector<float> o(a);
  o.insert(o.end(), b.begin(), b.end());
  return o;
}
// [2][64][64] k-major from a stacked [128][64] raw block: out[br][k][n] = raw[br*64+n][k]
static std::vector<float> branch_kmajor(const std::vector<float>& raw128x64) {
  std::vector<float> o(2 * 64 * 64);
  for (int br = 0; br < 2; br++)
    for (int k = 0; k < 64; k++)
      for (int n = 0; n < 64; n++) o[((size_t)br * 64 + k) * 64 + n] = raw128x64[((size_t)br * 64 + n) * 64 + k];
  return o;
}

// tf32 "hi" part: round-to-nearest (ties away) on the 13 dropped mantissa bits == cvt.rna.tf32.f32
static float tf32_hi_host(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u += 0x1000u;
  u &= 0xFFFFE000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}
// raw [N][K] row-major (K contiguous == K-major operand) -> canonical no-swizzle core-matrix layout
// (8 rows x 16 B per core matrix; K-chunk-major then row-group), hi plane followed by lo plane.
// element (n, k) at ((k/4) * (N/8) + n/8) * 32 + (n%8)*4 + k%4 ;  Kpad >= K pads with zeros.
static std::vector<float> canon_split(const std::vector<float>& raw, int N, int K, int Kpad) {
  std::vector<float> o((size_t)2 * N * Kpad, 0.f);
  for (int n = 0; n < N; n++)
    for (int k = 0; k < K; k++) {
      const size_t off = ((size_t)(k / 4) * (N / 8) + n / 8) * 32 + (n % 8) * 4 + (k % 4);
      const float x = raw[(size_t)n * K + k];
      const float h = tf32_hi_host(x);
      o[off] = h;
      o[(size_t)N * Kpad + off] = x - h;
    }
  return o;
}

static void finalize_weights(b2m_engine* e) {
  const int nb = e->desc.n_blocks;
  for (auto& kv : e->host_w) {
    const std::string& k = kv.first;
    bool bad = k.find("atom_graph_layers") != std::string::npos &&
               (k.find("edge_update_func") != std::string::npos || k.find("weight_func") != std::string::npos);
    bad = bad || (k.find("bond_graph_layers") != std::string::npos && k.find("weight_func") != std::string::npos);
    bad = bad || k.find("state_embedding") != std::string::npos || k.find("normalization") != std::string::npos;
    B2M_REQUIRE(!bad, B2M_ERR_INVALID,
                "unsupported CHGNet option (bond_update_hidden_dims / layer_bond_weights / state / norm): " + k);
  }
  e->consumed.clear();
  Packer P;
  std::map<std::string, size_t> off;
  std::vector<std::string> gemm_names;
  // every [K][N] row-major GEMM operand also gets a tcgen05 copy: canonical hi/lo planes of its [N][K] view
  auto put = [&](const std::string& name, const std::vector<float>& v) {
    off[name] = P.add(v);
    const bool is_k = name.size() > 2 && name.substr(name.size() - 2) == "_k";
    const bool is_raw = name.size() > 4 && name.substr(name.size() - 4) == "_raw";
    const bool is_f = name == "F0k" || name == "F1k" || name == "F0raw" || name == "F1raw";
    if ((is_k || is_raw || is_f) && name.find("Wg_k") == std::string::npos && name.find("WAg_k") == std::string::npos) {
      int K = 0, N = 0;
      if (v.size() == 64 * 64) K = 64, N = 64;
      else if (v.size() == 64 * 128) {
        // "_k" arrays of the first layers are [64][128]; "_raw" first-layer blocks are [128][64]
        if (is_raw) K = 128, N = 64; else K = 64, N = 128;
      }
      if (K) {
        off[name + ".can"] = P.add(canon_split(transpose(v, K, N), N, K, K));
        gemm_names.push_back(name);
      }
    }
  };

  const auto& f2 = W(e, "bond_expansion.frequencies", {NR});
  const auto& f3 = W(e, "threebody_bond_expansion.frequencies", {NR});
  const auto& fa = W(e, "angle_expansion.frequencies", {5});
  for (int k = 0; k < NR; k++) {
    e->rp2.freq[k] = f2[k];
    e->rp3.freq[k] = f3[k];
  }
  e->rp2.rc = (float)e->desc.cutoff;
  e->rp3.rc = (float)e->desc.three_body_cutoff;
  e->rp2.norm = (float)std::sqrt(2.0 / e->desc.cutoff);
  e->rp3.norm = (float)std::sqrt(2.0 / e->desc.three_body_cutoff);
  e->rp2.p = e->rp3.p = e->desc.cutoff_exponent;
  put("fa", fa);
  put("emb", W(e, "atom_embedding.weight", {e->desc.n_elem, D}));
  const auto& Wbe = W(e, "bond_embedding.layers.0.weight", {D, NR});
  put("Wbe", Wbe);
  put("Wae", W(e, "angle_embedding.layers.0.weight", {D, NF}));
  put("Wabw", W(e, "atom_bond_weights.weight", {D, NR}));
  put("W3bw", W(e, "threebody_bond_weights.weight", {D, NR}));

  for (int l = 0; l < nb; l++) {
    const std::string p = "atom_graph_layers." + std::to_string(l) + ".conv_layer.";
    const auto W1 = vcat(W(e, p + "node_update_func.layers.layers.0.weight", {D, 3 * D}),
                         W(e, p + "node_update_func.gates.layers.0.weight", {D, 3 * D}));  // [128][192]
    const auto b1 = vcat(W(e, p + "node_update_func.layers.layers.0.bias", {D}),
                         W(e, p + "node_update_func.gates.layers.0.bias", {D}));
    const auto W1s = cols(W1, 128, 192, 0), W1e = cols(W1, 128, 192, 64), W1t = cols(W1, 128, 192, 128);
    const auto W2 = vcat(W(e, p + "node_update_func.layers.layers.1.weight", {D, D}),
                         W(e, p + "node_update_func.gates.layers.1.weight", {D, D}));
    const auto b2 = vcat(W(e, p + "node_update_func.layers.layers.1.bias", {D}),
                         W(e, p + "node_update_func.gates.layers.1.bias", {D}));
    const auto& Wout = W(e, p + "node_out_func.weight", {D, D});
    std::vector<float> M(128 * 9);
    for (int j = 0; j < 128; j++)
      for (int k = 0; k < 9; k++) {
        double s = 0;
        for (int c = 0; c < 64; c++) s += (double)W1e[(size_t)j * 64 + c] * (double)Wbe[(size_t)c * 9 + k];
        M[j * 9 + k] = (float)s;
      }
    const std::string q = "a" + std::to_string(l) + ".";
    put(q + "W1s_k", transpose(W1s, 128, 64));
    put(q + "W1e_k", transpose(W1e, 128, 64));
    put(q + "W1t_k", transpose(W1t, 128, 64));
    put(q + "b1", b1);
    put(q + "W1s_raw", W1s);
    put(q + "W1e_raw", W1e);
    put(q + "W1t_raw", W1t);
    put(q + "M", M);
    put(q + "W2k", branch_kmajor(W2));
    put(q + "W2raw", W2);
    put(q + "b2", b2);
    put(q + "Wout_k", transpose(Wout, 64, 64));
    put(q + "Wout_raw", Wout);
    {
      const std::vector<float> W2L(W2.begin(), W2.begin() + 4096), W2G(W2.begin() + 4096, W2.end());
      put(q + "W2can", vcat(canon_split(W2L, 64, 64, 64), canon_split(W2G, 64, 64, 64)));
      put(q + "Mcan", canon_split(M, 128, 9, 16));
      put(q + "W2Tcan", vcat(canon_split(transpose(W2L, 64, 64), 64, 64, 64), canon_split(transpose(W2G, 64, 64), 64, 64, 64)));
    }
  }
  for (int l = 0; l < nb - 1; l++) {
    const std::string p = "bond_graph_layers." + std::to_string(l) + ".conv_layer.";
    const auto W1 = vcat(W(e, p + "node_update_func.layers.layers.0.weight", {D, 4 * D}),
                         W(e, p + "node_update_func.gates.layers.0.weight", {D, 4 * D}));  // [128][256]
    const auto b1 = vcat(W(e, p + "node_update_func.layers.layers.0.bias", {D}),
                         W(e, p + "node_update_func.gates.layers.0.bias", {D}));
    const auto W1a = cols(W1, 128, 256, 0), W1g = cols(W1, 128, 256, 64), W1c = cols(W1, 128, 256, 128),
               W1b = cols(W1, 128, 256, 192);
    const auto W2 = vcat(W(e, p + "node_update_func.layers.layers.1.weight", {D, D}),
                         W(e, p + "node_update_func.gates.layers.1.weight", {D, D}));
    const auto b2 = vcat(W(e, p + "node_update_func.layers.layers.1.bias", {D}),
                         W(e, p + "node_update_func.gates.layers.1.bias", {D}));
    const auto& Wout = W(e, p + "node_out_func.weight", {D, D});
    const auto WA = vcat(W(e, p + "edge_update_func.layers.layers.0.weight", {D, 4 * D}),
                         W(e, p + "edge_update_func.gates.layers.0.weight", {D, 4 * D}));
    const auto bA = vcat(W(e, p + "edge_update_func.layers.layers.0.bias", {D}),
                         W(e, p + "edge_update_func.gates.layers.0.bias", {D}));
    const auto WAa = cols(WA, 128, 256, 0), WAg = cols(WA, 128, 256, 64), WAc = cols(WA, 128, 256, 128),
               WAb = cols(WA, 128, 256, 192);
    const std::string q = "b" + std::to_string(l) + ".";
    put(q + "W1a_k", transpose(W1a, 128, 64));
    put(q + "W1b_k", transpose(W1b, 128, 64));
    put(q + "W1c_k", transpose(W1c, 128, 64));
    put(q + "Wg_k", branch_kmajor(W1g));
    put(q + "b1", b1);
    put(q + "W1a_raw", W1a);
    put(q + "W1b_raw", W1b);
    put(q + "W1c_raw", W1c);
    put(q + "Wg_raw", W1g);
    put(q + "W2k", branch_kmajor(W2));
    put(q + "W2raw", W2);
    put(q + "b2", b2);
    put(q + "Wout_k", transpose(Wout, 64, 64));
    put(q + "Wout_raw", Wout);
    put(q + "WAa_k", transpose(WAa, 128, 64));
    put(q + "WAb_k", transpose(WAb, 128, 64));
    put(q + "WAc_k", transpose(WAc, 128, 64));
    put(q + "WAg_k", branch_kmajor(WAg));
    put(q + "bA", bA);
    put(q + "WAa_raw", WAa);
    put(q + "WAb_raw", WAb);
    put(q + "WAc_raw", WAc);
    put(q + "WAg_raw", WAg);
    {
      auto rows64 = [](const std::vector<float>& m, int br) {
        return std::vector<float>(m.begin() + (size_t)br * 4096, m.begin() + (size_t)(br + 1) * 4096);
      };
      const std::vector<float> W2L(W2.begin(), W2.begin() + 4096), W2G(W2.begin() + 4096, W2.end());
      put(q + "Wgcan", canon_split(W1g, 128, 64, 64));
      put(q + "W2can", vcat(canon_split(W2L, 64, 64, 64), canon_split(W2G, 64, 64, 64)));
      put(q + "W2Tcan", vcat(canon_split(transpose(W2L, 64, 64), 64, 64, 64), canon_split(transpose(W2G, 64, 64), 64, 64, 64)));
      put(q + "WgTcan", vcat(canon_split(transpose(rows64(W1g, 0), 64, 64), 64, 64, 64),
                             canon_split(transpose(rows64(W1g, 1), 64, 64), 64, 64, 64)));
      put(q + "WAgcan", canon_split(WAg, 128, 64, 64));
      put(q + "WAgTcan", vcat(canon_split(transpose(rows64(WAg, 0), 64, 64), 64, 64, 64),
                              canon_split(transpose(rows64(WAg, 1), 64, 64), 64, 64, 64)));
    }
  }
  const auto& F0 = W(e, "final_layer.layers.0.weight", {D, D});
  const auto& F1 = W(e, "final_layer.layers.1.weight", {D, D});
  put("F0k", transpose(F0, 64, 64));
  put("F0raw", F0);
  put("c0", W(e, "final_layer.layers.0.bias", {D}));
  put("F1k", transpose(F1, 64, 64));
  put("F1raw", F1);
  put("c1", W(e, "final_layer.layers.1.bias", {D}));
  put("F2", W(e, "final_layer.layers.2.weight", {1, D}));
  e->c2 = W(e, "final_layer.layers.2.bias", {1})[0];
  put("Ws", W(e, "sitewise_readout.weight", {1, D}));
  e->bs = W(e, "sitewise_readout.bias", {1})[0];
  // every tensor of the state_dict must have been used: an extra bias / normalisation / per-layer weight function of
  // a non-default CHGNet configuration would otherwise be dropped silently and give wrong energies (ADVICE r1).
  // bond_bond_weights is part of the default model but feeds only the (absent) bond update of the atom graph.
  for (auto& kv : e->host_w) {
    if (e->consumed.count(kv.first) || kv.first == "bond_bond_weights.weight") continue;
    throw Error(B2M_ERR_INVALID, "state_dict tensor '" + kv.first +
                                     "' is not used by this engine (unsupported CHGNet configuration; refusing to ignore it)");
  }
  if (!e->elem_refs.empty()) {
    e->erefbuf.ensure(e->elem_refs.size());
    B2M_CK(cudaMemcpyAsync(e->erefbuf.p, e->elem_refs.data(), e->elem_refs.size() * sizeof(double), cudaMemcpyHostToDevice,
                           e->st));
  }
  e->wbuf.ensure(P.host.size() + 64);
  B2M_CK(cudaMemcpyAsync(e->wbuf.p, P.host.data(), P.host.size() * sizeof(float), cudaMemcpyHostToDevice, e->st));
  B2M_CK(cudaStreamSynchronize(e->st));
  auto dp = [&](const std::string& n) { return e->wbuf.p + off.at(n); };
  e->canon_of.clear();
  for (auto& n : gemm_names) e->canon_of[dp(n)] = dp(n + ".can");
  e->d_fa = dp("fa");
  e->d_emb = dp("emb");
  e->d_Wbe = dp("Wbe");
  e->d_Wae = dp("Wae");
  e->d_Wabw = dp("Wabw");
  e->d_W3bw = dp("W3bw");
  e->d_F0k = dp("F0k"), e->d_F0raw = dp("F0raw"), e->d_c0 = dp("c0");
  e->d_F1k = dp("F1k"), e->d_F1raw = dp("F1raw"), e->d_c1 = dp("c1");
  e->d_F2 = dp("F2"), e->d_Ws = dp("Ws");
  e->d_eref = e->elem_refs.empty() ? nullptr : e->erefbuf.p;
  e->aw.resize(nb);
  for (int l = 0; l < nb; l++) {
    const std::string q = "a" + std::to_string(l) + ".";
    AtomLayerW& w = e->aw[l];
    w.W1s_k = dp(q + "W1s_k"), w.W1e_k = dp(q + "W1e_k"), w.W1t_k = dp(q + "W1t_k"), w.b1 = dp(q + "b1");
    w.W1s_raw = dp(q + "W1s_raw"), w.W1e_raw = dp(q + "W1e_raw"), w.W1t_raw = dp(q + "W1t_raw");
    w.M = dp(q + "M"), w.W2k = dp(q + "W2k"), w.W2raw = dp(q + "W2raw"), w.b2 = dp(q + "b2");
    w.Wout_k = dp(q + "Wout_k"), w.Wout_raw = dp(q + "Wout_raw");
    w.W2can = dp(q + "W2can"), w.Mcan = dp(q + "Mcan"), w.W2Tcan = dp(q + "W2Tcan");
  }
  e->bw.resize(nb - 1);
  for (int l = 0; l < nb - 1; l++) {
    const std::string q = "b" + std::to_string(l) + ".";
    BondLayerW& w = e->bw[l];
    w.W1a_k = dp(q + "W1a_k"), w.W1b_k = dp(q + "W1b_k"), w.W1c_k = dp(q + "W1c_k"), w.Wg_k = dp(q + "Wg_k");
    w.b1 = dp(q + "b1"), w.W1a_raw = dp(q + "W1a_raw"), w.W1b_raw = dp(q + "W1b_raw"), w.W1c_raw = dp(q + "W1c_raw");
    w.Wg_raw = dp(q + "Wg_raw"), w.W2k = dp(q + "W2k"), w.W2raw = dp(q + "W2raw"), w.b2 = dp(q + "b2");
    w.Wout_k = dp(q + "Wout_k"), w.Wout_raw = dp(q + "Wout_raw");
    w.WAa_k = dp(q + "WAa_k"), w.WAb_k = dp(q + "WAb_k"), w.WAc_k = dp(q + "WAc_k"), w.WAg_k = dp(q + "WAg_k");
    w.bA = dp(q + "bA"), w.WAa_raw = dp(q + "WAa_raw"), w.WAb_raw = dp(q + "WAb_raw"), w.WAc_raw = dp(q + "WAc_raw");
    w.WAg_raw = dp(q + "WAg_raw");
    w.Wgcan = dp(q + "Wgcan"), w.W2can = dp(q + "W2can"), w.W2Tcan = dp(q + "W2Tcan"), w.WgTcan = dp(q + "WgTcan");
    w.WAgcan = dp(q + "WAgcan"), w.WAgTcan = dp(q + "WAgTcan");
  }
  e->finalized = true;
}

// node-level GEMM dispatch: tcgen05 when a canonical copy of B exists, FFMA tile kernel otherwise
static void gemm(b2m_engine* e, const float* A, int lda, const float* B, float* C, int ldc, int M, int N, int K,
                 const float* bias, const float* R, int ldr, bool accum) {
  if (e->use_tc) {
    auto it = e->canon_of.find(B);
    if (it != e->canon_of.end()) {
      launch_gemm_tc(e->st, A, lda, it->second, C, ldc, M, N, K, bias, R, ldr, accum, e->num_sms);
      return;
    }
  }
  B2M_REQUIRE(!e->use_tc, B2M_ERR_STATE, "tcgen05 path: GEMM operand without a canonical copy");
  launch_gemm(e->st, A, lda, B, C, ldc, M, N, K, bias, R, ldr, accum);  // FP32-FFMA tile kernel (legacy path only)
}

// ------------------------------------------------------------------------------------------
static void alloc_workspace(b2m_engine* e) {
  Graph& g = e->g;
  const int nb = e->desc.n_blocks;
  const size_t nl = g.n_loc, no = g.n_own, bl = g.B_loc, bo = g.B_own;
  const size_t A = (size_t)g.A, E = (size_t)g.E;
  e->x.resize(nb + 1);
  e->h.resize(nb);
  e->ang.resize(nb - 1);
  e->upd.resize(nb - 1);
  for (auto& b : e->x) b.ensure(nl * D + 64);
  for (auto& b : e->h) b.ensure(bl * D + 64);
  const size_t Apad = (A + 127) / 128 * 128;  // tile-interleaved on the tcgen05 path: whole tiles
  for (auto& b : e->ang) b.ensure(Apad * D + 64);
  for (auto& b : e->upd) b.ensure(bo * D + 64);
  e->uv.resize(nb);
  if (e->use_tc)
    for (auto& b : e->uv) b.ensure(((E + 127) / 128 * 128) * D2 + 64);  // u|v kept for the backward (tile-interleaved)
  e->uvB.resize(nb - 1), e->dsB.resize(nb - 1), e->uvA.resize(nb - 1);
  if (e->use_tc) {
    e->be_e.ensure(((E + 127) / 128 * 128) * 12 + 64), e->dbe_e.ensure(((E + 127) / 128 * 128) * 12 + 64);
    const size_t Ap = (A + 127) / 128 * 128;
    for (auto& b : e->uvB) b.ensure(Ap * D2 + 64);
    for (auto& b : e->dsB) b.ensure(Ap * D2 + 64);
    for (int l = 0; l < nb - 2; l++) e->uvA[l].ensure(Ap * D2 + 64);
  }
  e->ApL.resize(nb), e->CpL.resize(nb), e->QpL.resize(nb);
  for (int l = 0; l < nb; l++) {
    e->ApL[l].ensure(nl * D2 + 64), e->CpL[l].ensure(no * D2 + 64);
    if (l > 0) e->QpL[l].ensure(bo * D2 + 64);
  }
  e->Ha.ensure(bl * D2 + 64), e->Hb.ensure(bo * D2 + 64), e->Xc.ensure(nl * D2 + 64);
  e->agg.ensure(no * D + 64), e->aggB.ensure(bo * D + 64);
  e->y1p.ensure(no * D), e->y1.ensure(no * D), e->y2p.ensure(no * D), e->y2.ensure(no * D);
  e->e_atom.ensure(no), e->site.ensure(no);
  e->gx.ensure(nl * D + 64), e->gh.ensure(bl * D + 64), e->gang.ensure(Apad * D + 64);
  e->gA.ensure(nl * D2 + 64), e->gC.ensure(no * D2 + 64), e->gQ.ensure(bo * D2 + 64);
  e->gHa.ensure(bl * D2 + 64), e->gHb.ensure(bo * D2 + 64), e->gXc.ensure(nl * D2 + 64);
  e->gagg.ensure(no * D + 64), e->gupd.ensure(bo * D + 64), e->gaggB.ensure(bo * D + 64);
  e->gd.ensure(E + 64), e->gdb.ensure(bl + 64), e->gbvec.ensure(bl * 3 + 64);
  e->gy1.ensure(no * D), e->gy2.ensure(no * D);
  e->forces.ensure((size_t)g.N * 3 + 64);
  e->site_full.ensure((size_t)g.N + 64);
  e->scal.ensure(16);
  if (e->world > 1) {
    size_t tot_to = 0, tot_bto = 0;
    for (int q = 0; q < e->world; q++) tot_to += g.n_to[q], tot_bto += g.nb_to[q];
    size_t m = std::max(tot_to * D, tot_bto * D);
    if (e->leader != nullptr) {
      e->precv[0].ensure(m + 64), e->precv[1].ensure(m + 64);
    } else {
      e->sendbuf.ensure(m + 64);
      e->recvbuf.ensure(m + 64);
    }
  }
}

// ---- halo exchange between slab neighbours ----
// Two transports: NCCL point-to-point (one process per GPU, world > 1 with a communicator) and, inside a single-process
// group, direct peer-memory traffic: the sender's pack kernel stores its boundary rows straight into the receiver's halo
// rows (forward) or copies its halo adjoints into the owner's receive buffer (backward); a CUDA event per exchange point
// orders the receiver's stream behind the sender's.
// kind 0: atom rows x[l] | 1: bond rows h[l] | 2: TensorNet atom tensors X[l] (10 x 64 floats per atom)
static float* halo_buffer(b2m_engine* e, int kind, int l) {
  return kind == 1 ? e->h[l].p : (kind == 2 ? e->tn->X[l].p : e->x[l].p);
}
static int halo_width(int kind) { return kind == 2 ? 10 * D : D; }

static cudaEvent_t next_halo_event(b2m_engine* e) {
  // the events are created in b2m_create: a neighbour's thread reads hev[k] concurrently, so the vector never grows here
  B2M_REQUIRE(e->hpoint < (int)e->hev.size(), B2M_ERR_STATE, "too many halo-exchange points in one evaluation");
  return e->hev[e->hpoint];
}

// forward: rows of tensor (bonds ? h : x)[l] listed in to_list[q] -> q's halo section; my halo section <- owners.
// Split in two so that the exchange runs on the engine's second stream while the compute stream does the projections
// that do not read the halo rows (the reference issues its copies on the compute stream, dist.py:344-356):
//   halo_forward_begin: [compute: producer done] -> [comm stream: pack, send / receive or peer stores]
//   halo_forward_end  : compute stream waits for the exchange (and, in a group, for the neighbours' stores)
static void halo_forward_begin(b2m_engine* e, int kind, int l) {
  if (e->world <= 1 || e->debug_no_halo) return;
  Graph& g = e->g;
  const bool bonds = kind == 1;
  const size_t W = (size_t)halo_width(kind);
  float* buf = halo_buffer(e, kind, l);
  const int* nto = bonds ? g.nb_to : g.n_to;
  const int* toff = bonds ? g.bto_off : g.to_off;
  const int* nfrom = bonds ? g.nb_from : g.n_from;
  const int* foff = bonds ? g.bfrom_off : g.from_off;
  const int* list = bonds ? g.bto_list.p : g.to_list.p;
  const size_t base = bonds ? (size_t)g.B_own : (size_t)g.n_own;
  B2M_CK(cudaEventRecord(e->ev_prod, e->st));
  B2M_CK(cudaStreamWaitEvent(e->cst, e->ev_prod, 0));
  if (e->leader != nullptr) {
    b2m_engine* L = e->leader;
    for (int q = 0; q < e->world; q++) {
      if (q == e->rank || nto[q] <= 0) continue;
      b2m_engine* pe = L->parts[q];
      Graph& pg = pe->g;
      const int pn = bonds ? pg.nb_from[e->rank] : pg.n_from[e->rank];
      B2M_REQUIRE(pn == nto[q], B2M_ERR_STATE, "halo sections of two partitions disagree");
      const size_t pbase = bonds ? (size_t)pg.B_own : (size_t)pg.n_own;
      const size_t pfoff = bonds ? (size_t)pg.bfrom_off[e->rank] : (size_t)pg.from_off[e->rank];
      launch_gather_rows(e->cst, nto[q], (int)W, list + toff[q], buf, halo_buffer(pe, kind, l) + (pbase + pfoff) * W);
    }
    B2M_CK(cudaEventRecord(next_halo_event(e), e->cst));
    return;
  }
  for (int q = 0; q < e->world; q++)
    if (nto[q] > 0)
      launch_gather_rows(e->cst, nto[q], (int)W, list + toff[q], buf, e->sendbuf.p + (size_t)toff[q] * W);
  NCCL_CK(g_nccl.GroupStart());
  for (int q = 0; q < e->world; q++) {
    if (q == e->rank) continue;
    if (nto[q] > 0)
      NCCL_CK(g_nccl.Send(e->sendbuf.p + (size_t)toff[q] * W, (size_t)nto[q] * W, ncclFloat32, q, e->comm, e->cst));
    if (nfrom[q] > 0)
      NCCL_CK(g_nccl.Recv(buf + (base + foff[q]) * W, (size_t)nfrom[q] * W, ncclFloat32, q, e->comm, e->cst));
  }
  NCCL_CK(g_nccl.GroupEnd());
  B2M_CK(cudaEventRecord(e->ev_halo, e->cst));
}
static void halo_forward_end(b2m_engine* e) {
  if (e->world <= 1 || e->debug_no_halo) return;
  if (e->leader != nullptr) {
    b2m_engine* L = e->leader;
    const int k = e->hpoint++;
    L->gsync.arrive_and_wait();  // every partition has recorded its event for this point
    for (int q = 0; q < e->world; q++)  // own event too: my stores must precede any later reuse of the source rows
      B2M_CK(cudaStreamWaitEvent(e->st, L->parts[q]->hev[k], 0));
    return;
  }
  B2M_CK(cudaStreamWaitEvent(e->st, e->ev_halo, 0));
}
// backward: my halo rows of the adjoint -> owners (accumulate), then zero the halo rows
static void halo_backward(b2m_engine* e, float* gbuf, bool bonds, int width = D) {
  if (e->world <= 1 || e->debug_no_halo) return;
  Graph& g = e->g;
  const size_t W = (size_t)width;
  const int* nto = bonds ? g.nb_to : g.n_to;
  const int* toff = bonds ? g.bto_off : g.to_off;
  const int* nfrom = bonds ? g.nb_from : g.n_from;
  const int* foff = bonds ? g.bfrom_off : g.from_off;
  const int* list = bonds ? g.bto_list.p : g.to_list.p;
  const size_t base = bonds ? (size_t)g.B_own : (size_t)g.n_own;
  const size_t nhalo = bonds ? (size_t)g.B_halo : (size_t)g.n_halo;
  if (e->leader != nullptr) {
    b2m_engine* L = e->leader;
    const int k = e->hpoint;
    for (int q = 0; q < e->world; q++) {
      if (q == e->rank || nfrom[q] <= 0) continue;
      b2m_engine* pe = L->parts[q];
      const size_t ptoff = bonds ? (size_t)pe->g.bto_off[e->rank] : (size_t)pe->g.to_off[e->rank];
      // the owner's receive buffer of this parity was consumed two exchange points ago (see DESIGN.md, group mode)
      B2M_CK(cudaMemcpyAsync(pe->precv[k & 1].p + ptoff * W, gbuf + (base + foff[q]) * W, (size_t)nfrom[q] * W * sizeof(float),
                             cudaMemcpyDefault, e->st));
    }
    launch_zero_rows(e->st, gbuf + base * W, nhalo * W);
    cudaEvent_t ev = next_halo_event(e);
    B2M_CK(cudaEventRecord(ev, e->st));
    e->hpoint++;
    L->gsync.arrive_and_wait();
    for (int q = 0; q < e->world; q++)
      if (q != e->rank) B2M_CK(cudaStreamWaitEvent(e->st, L->parts[q]->hev[k], 0));
    for (int q = 0; q < e->world; q++)
      if (q != e->rank && nto[q] > 0)
        launch_scatter_add_rows(e->st, nto[q], (int)W, list + toff[q], e->precv[k & 1].p + (size_t)toff[q] * W, gbuf);
    return;
  }
  NCCL_CK(g_nccl.GroupStart());
  for (int q = 0; q < e->world; q++) {
    if (q == e->rank) continue;
    if (nfrom[q] > 0)
      NCCL_CK(g_nccl.Send(gbuf + (base + foff[q]) * W, (size_t)nfrom[q] * W, ncclFloat32, q, e->comm, e->st));
    if (nto[q] > 0)
      NCCL_CK(g_nccl.Recv(e->recvbuf.p + (size_t)toff[q] * W, (size_t)nto[q] * W, ncclFloat32, q, e->comm, e->st));
  }
  NCCL_CK(g_nccl.GroupEnd());
  for (int q = 0; q < e->world; q++)
    if (nto[q] > 0)
      launch_scatter_add_rows(e->st, nto[q], (int)W, list + toff[q], e->recvbuf.p + (size_t)toff[q] * W, gbuf);
  launch_zero_rows(e->st, gbuf + base * W, nhalo * W);
}

#include "engine_tn.inl"

static AtomConvArgs atom_args(b2m_engine* e, int l) {
  Graph& g = e->g;
  const AtomLayerW& w = e->aw[l];
  AtomConvArgs a;
  memset(&a, 0, sizeof a);
  a.E = g.E;
  a.e_src = g.e_src.p, a.e_dst = g.e_dst.p, a.e_bond = g.e_bond.p, a.e_vec = g.e_vec.p;
  const int ps = e->proj_slot(l);
  a.Aproj = e->ApL[ps].p, a.Cproj = e->CpL[ps].p, a.Qproj = l > 0 ? e->QpL[ps].p : nullptr;
  a.M = w.M, a.W2k = w.W2k, a.W2raw = w.W2raw, a.b2 = w.b2, a.Wabw = e->d_Wabw;
  a.rp = e->rp2;
  a.be = e->be_e.p, a.dbe = e->dbe_e.p;
  return a;
}
static void atom_projections(b2m_engine* e, int l) {
  Graph& g = e->g;
  const AtomLayerW& w = e->aw[l];
  const int ps = e->proj_slot(l);
  gemm(e, e->x[l].p, D, w.W1s_k, e->ApL[ps].p, D2, g.n_loc, D2, D, nullptr, nullptr, 0, false);
  gemm(e, e->x[l].p, D, w.W1t_k, e->CpL[ps].p, D2, g.n_own, D2, D, w.b1, nullptr, 0, false);
  if (l > 0) gemm(e, e->h[l].p, D, w.W1e_k, e->QpL[ps].p, D2, g.B_own, D2, D, nullptr, nullptr, 0, false);
}
static void atom_layer_fwd(b2m_engine* e, int l) {
  Graph& g = e->g;
  const AtomLayerW& w = e->aw[l];
  atom_projections(e, l);
  launch_zero_rows(e->st, e->agg.p, (int64_t)g.n_own * D);
  AtomConvArgs a = atom_args(e, l);
  a.agg = e->agg.p;
  cudaEvent_t e0, e1;
  B2M_CK(cudaEventCreate(&e0));
  B2M_CK(cudaEventCreate(&e1));
  B2M_CK(cudaEventRecord(e0, e->st));
  if (e->use_tc) {
    AtomConvTcW tw{w.W2can, w.Mcan, w.W2Tcan};
    a.uv_save = e->want_grads ? e->uv[l].p : nullptr;
    if (e->ac_gen >= 3)
      launch_atomconv_fwd_v3(e->st, a, tw, e->num_sms);
    else
      launch_atomconv_fwd_tc(e->st, a, tw, e->num_sms);
  } else {
    launch_atomconv_fwd(e->st, a);
  }
  B2M_CK(cudaEventRecord(e1, e->st));
  e->gather_ev.push_back({e0, e1});
  gemm(e, e->agg.p, D, w.Wout_k, e->x[l + 1].p, D, g.n_own, D, D, nullptr, e->x[l].p, D, false);
}
// in: gx = dE/dx[l+1] (owned rows valid, halo rows zero).  out: gx = dE/dx[l] (all local rows)
static void atom_layer_bwd(b2m_engine* e, int l) {
  Graph& g = e->g;
  const AtomLayerW& w = e->aw[l];
  gemm(e, e->gx.p, D, w.Wout_raw, e->gagg.p, D, g.n_own, D, D, nullptr, nullptr, 0, false);
  // A / C / Q of this layer are still in their per-layer buffers from the forward: no recompute
  AtomConvArgs a = atom_args(e, l);
  a.gagg = e->gagg.p;
  a.gd = e->gd.p;
  const bool need_gx = l > 0;
  if (need_gx) {
    launch_zero_rows(e->st, e->gA.p, (int64_t)g.n_loc * D2);
    launch_zero_rows(e->st, e->gC.p, (int64_t)g.n_own * D2);
    a.gA = e->gA.p, a.gC = e->gC.p, a.gQ = e->gQ.p;
  }
  if (e->use_tc) {
    AtomConvTcW tw{w.W2can, w.Mcan, w.W2Tcan};
    a.uv = e->uv[l].p;
    if (e->ac_gen >= 3 && e->ac_gen != 4)  // B2M_ATOMCONV=4: third-generation forward with the first-generation backward
      launch_atomconv_bwd_v3(e->st, a, tw, e->num_sms);
    else
      launch_atomconv_bwd_tc(e->st, a, tw, e->num_sms);
  } else {
    launch_atomconv_bwd(e->st, a);
  }
  if (need_gx) {
    gemm(e, e->gA.p, D2, w.W1s_raw, e->gx.p, D, g.n_loc, D, D2, nullptr, nullptr, 0, true);
    gemm(e, e->gC.p, D2, w.W1t_raw, e->gx.p, D, g.n_own, D, D2, nullptr, nullptr, 0, true);
    gemm(e, e->gQ.p, D2, w.W1e_raw, e->gh.p, D, g.B_own, D, D2, nullptr, nullptr, 0, true);
  }
}

static LineArgs line_args(b2m_engine* e, int l, bool hidden) {
  Graph& g = e->g;
  const BondLayerW& w = e->bw[l];
  LineArgs a;
  memset(&a, 0, sizeof a);
  a.A = g.A;
  a.a_in = g.a_in.p, a.a_out = g.a_out.p, a.a_ctr = g.a_ctr.p;
  a.ang = e->ang[l].p;
  a.Ha = e->Ha.p, a.Hb = e->Hb.p, a.Xc = e->Xc.p;
  if (hidden) {
    a.Wgk = w.Wg_k, a.Wgraw = w.Wg_raw, a.W2k = w.W2k, a.W2raw = w.W2raw, a.b2 = w.b2;
  } else {
    a.Wgk = w.WAg_k, a.Wgraw = w.WAg_raw;
  }
  if (e->use_tc) {
    float* uvp = hidden ? e->uvB[l].p : e->uvA[l].p;
    a.uv = uvp, a.ds = hidden ? e->dsB[l].p : nullptr;
    if (e->want_grads) a.uv_save = uvp, a.ds_save = hidden ? e->dsB[l].p : nullptr;
  }
  return a;
}
static LineTcW line_tcw(b2m_engine* e, int l, bool hidden) {
  const BondLayerW& w = e->bw[l];
  LineTcW t;
  if (hidden) {
    t.Wgcan = w.Wgcan, t.W2can = w.W2can, t.W2Tcan = w.W2Tcan, t.WgTcan = w.WgTcan;
  } else {
    t.Wgcan = w.WAgcan, t.W2can = nullptr, t.W2Tcan = nullptr, t.WgTcan = w.WAgTcan;
  }
  return t;
}
static void line_fwd_dispatch(b2m_engine* e, int l, bool hidden, const LineArgs& a) {
  if (e->use_tc)
    launch_line_fwd_tc(e->st, a, line_tcw(e, l, hidden), hidden, e->num_sms);
  else
    launch_line_fwd(e->st, a, hidden);
}
// first-layer projections of the line-graph MLPs: Ha / Hb from the bond features, Xc from the atom features
static void line_proj_Ha(b2m_engine* e, int l, bool hidden) {
  const BondLayerW& w = e->bw[l];
  const float* hsrc = hidden ? e->h[l].p : e->h[l + 1].p;
  gemm(e, hsrc, D, hidden ? w.W1a_k : w.WAa_k, e->Ha.p, D2, e->g.B_loc, D2, D, nullptr, nullptr, 0, false);
}
static void line_proj_Hb(b2m_engine* e, int l, bool hidden) {
  const BondLayerW& w = e->bw[l];
  const float* hsrc = hidden ? e->h[l].p : e->h[l + 1].p;
  gemm(e, hsrc, D, hidden ? w.W1b_k : w.WAb_k, e->Hb.p, D2, e->g.B_own, D2, D, hidden ? w.b1 : w.bA, nullptr, 0, false);
}
static void line_proj_Xc(b2m_engine* e, int l, bool hidden) {
  const BondLayerW& w = e->bw[l];
  gemm(e, e->x[l + 1].p, D, hidden ? w.W1c_k : w.WAc_k, e->Xc.p, D2, e->g.n_loc, D2, D, nullptr, nullptr, 0, false);
}
static void line_projections(b2m_engine* e, int l, bool hidden) {
  line_proj_Ha(e, l, hidden), line_proj_Hb(e, l, hidden), line_proj_Xc(e, l, hidden);
}
static void line_bwd_common(b2m_engine* e, int l, bool hidden, LineArgs& a) {
  Graph& g = e->g;
  const BondLayerW& w = e->bw[l];
  launch_zero_rows(e->st, e->gHa.p, (int64_t)g.B_loc * D2);
  launch_zero_rows(e->st, e->gHb.p, (int64_t)g.B_own * D2);
  launch_zero_rows(e->st, e->gXc.p, (int64_t)g.n_loc * D2);
  a.gang = e->gang.p, a.gHa = e->gHa.p, a.gHb = e->gHb.p, a.gXc = e->gXc.p;
  if (e->use_tc)
    launch_line_bwd_tc(e->st, a, line_tcw(e, l, hidden), hidden, e->num_sms);
  else
    launch_line_bwd(e->st, a, hidden);
  gemm(e, e->gHa.p, D2, hidden ? w.W1a_raw : w.WAa_raw, e->gh.p, D, g.B_loc, D, D2, nullptr, nullptr, 0, true);
  gemm(e, e->gHb.p, D2, hidden ? w.W1b_raw : w.WAb_raw, e->gh.p, D, g.B_own, D, D2, nullptr, nullptr, 0, true);
  gemm(e, e->gXc.p, D2, hidden ? w.W1c_raw : w.WAc_raw, e->gx.p, D, g.n_loc, D, D2, nullptr, nullptr, 0, true);
}

static void forward(b2m_engine* e) {
  Graph& g = e->g;
  const int nb = e->desc.n_blocks;
  if (e->use_tc) launch_edge_basis(e->st, g.E, g.e_vec.p, e->rp2, e->be_e.p, e->dbe_e.p);
  launch_embed(e->st, g.n_loc, g.type.p, e->d_emb, e->x[0].p);
  launch_bond_init(e->st, g.B_loc, g.b_vec.p, e->rp2, e->d_Wbe, e->h[0].p);
  launch_angle_init(e->st, g.A, g.a_in.p, g.a_out.p, g.b_vec.p, e->d_fa, e->d_Wae, e->ang[0].p, e->use_tc);
  for (int l = 0; l < nb - 1; l++) {
    atom_layer_fwd(e, l);
    const BondLayerW& w = e->bw[l];
    // x^{l+1} halo rows travel while the two projections of the bond features run (they do not read x)
    halo_forward_begin(e, false, l + 1);
    line_proj_Ha(e, l, true), line_proj_Hb(e, l, true);
    halo_forward_end(e);
    line_proj_Xc(e, l, true);
    launch_zero_rows(e->st, e->aggB.p, (int64_t)g.B_own * D);
    LineArgs a = line_args(e, l, true);
    a.aggB = e->aggB.p;
    line_fwd_dispatch(e, l, true, a);
    gemm(e, e->aggB.p, D, w.Wout_k, e->upd[l].p, D, g.B_own, D, D, nullptr, nullptr, 0, false);
    launch_bond_update_fwd(e->st, g.B_own, g.b_vec.p, e->rp3, e->d_W3bw, e->h[l].p, e->upd[l].p, e->h[l + 1].p);
    if (l < nb - 2) {
      // the last block's angle update (and the halo copy of h feeding it) is dead code in the
      // reference (chgnet.py:353-368 on the last iteration): nothing reads it afterwards.
      // h^{l+1} halo rows travel while Hb (owned bonds only) and Xc (atoms) are projected; Ha reads the halo rows
      halo_forward_begin(e, true, l + 1);
      line_proj_Hb(e, l, false), line_proj_Xc(e, l, false);
      halo_forward_end(e);
      line_proj_Ha(e, l, false);
      LineArgs b = line_args(e, l, false);
      b.ang_out = e->ang[l + 1].p;
      line_fwd_dispatch(e, l, false, b);
    }
  }
  // site-wise readout after block n-2 (chgnet.py:392-398)
  launch_rowdot(e->st, g.n_own, e->x[nb - 1].p, e->d_Ws, e->bs, e->site.p, nullptr, nullptr, nullptr, 1.f);
  atom_layer_fwd(e, nb - 1);
  // final MLP 64 -> 64 -> 64 -> 1, sum (chgnet.py:422-440); E = std * E + mean (+ element refs) (pes.py:109-113)
  gemm(e, e->x[nb].p, D, e->d_F0k, e->y1p.p, D, g.n_own, D, D, e->d_c0, nullptr, 0, false);
  launch_silu(e->st, (int64_t)g.n_own * D, e->y1p.p, e->y1.p);
  gemm(e, e->y1.p, D, e->d_F1k, e->y2p.p, D, g.n_own, D, D, e->d_c1, nullptr, 0, false);
  launch_silu(e->st, (int64_t)g.n_own * D, e->y2p.p, e->y2.p);
  B2M_CK(cudaMemsetAsync(e->scal.p, 0, 16 * sizeof(double), e->st));
  launch_rowdot(e->st, g.n_own, e->y2.p, e->d_F2, e->c2, e->e_atom.p, e->scal.p, g.type.p, e->d_eref,
                (float)e->desc.data_std);
}

static void backward(b2m_engine* e) {
  Graph& g = e->g;
  const int nb = e->desc.n_blocks;
  launch_zero_rows(e->st, e->gd.p, g.E);
  launch_zero_rows(e->st, e->gdb.p, g.B_loc);
  launch_zero_rows(e->st, e->gbvec.p, (int64_t)g.B_loc * 3);
  launch_zero_rows(e->st, e->gh.p, (int64_t)g.B_loc * D);
  launch_zero_rows(e->st, e->gang.p, (g.A + 127) / 128 * 128 * D);
  launch_zero_rows(e->st, e->gx.p, (int64_t)g.n_loc * D);
  launch_zero_rows(e->st, e->forces.p, g.N * 3);
  // readout backward
  launch_readout_seed(e->st, g.n_own, e->y2p.p, e->d_F2, (float)e->desc.data_std, e->gy2.p);
  gemm(e, e->gy2.p, D, e->d_F1raw, e->gy1.p, D, g.n_own, D, D, nullptr, nullptr, 0, false);
  launch_dsilu_mul(e->st, (int64_t)g.n_own * D, e->y1p.p, e->gy1.p);
  gemm(e, e->gy1.p, D, e->d_F0raw, e->gx.p, D, g.n_own, D, D, nullptr, nullptr, 0, false);
  atom_layer_bwd(e, nb - 1);
  for (int l = nb - 2; l >= 0; l--) {
    const BondLayerW& w = e->bw[l];
    if (l < nb - 2) {
      // the tcgen05 backward works from the tensors saved by the forward; only the FFMA generation recomputes
      // the first-layer projections
      if (!e->use_tc) line_projections(e, l, false);
      LineArgs a = line_args(e, l, false);
      line_bwd_common(e, l, false, a);
      halo_backward(e, e->gh.p, true);
    }
    launch_bond_update_bwd(e->st, g.B_own, g.b_vec.p, e->rp3, e->d_W3bw, e->gh.p, e->upd[l].p, e->gupd.p, e->gdb.p);
    gemm(e, e->gupd.p, D, w.Wout_raw, e->gaggB.p, D, g.B_own, D, D, nullptr, nullptr, 0, false);
    if (!e->use_tc) line_projections(e, l, true);
    LineArgs a = line_args(e, l, true);
    a.gaggB = e->gaggB.p;
    line_bwd_common(e, l, true, a);
    halo_backward(e, e->gx.p, false);
    atom_layer_bwd(e, l);
  }
  // geometry: h0 = W_be be(d_b), theta/Fourier, then edges -> forces and virial
  launch_h0_bwd(e->st, g.B_loc, g.b_vec.p, e->rp2, e->d_Wbe, e->gh.p, e->gdb.p);
  launch_angle_init_bwd(e->st, g.A, g.a_in.p, g.a_out.p, g.b_vec.p, e->d_fa, e->d_Wae, e->gang.p, e->gbvec.p, e->use_tc);
  float* atom_vir = e->want_peratom ? e->atom_vir.p : nullptr;
  launch_edge_final(e->st, g.E, g.e_src.p, g.e_dst.p, g.e_bond.p, g.e_vec.p, g.gid.p, e->gd.p, e->gdb.p, e->gbvec.p,
                    e->forces.p, e->scal.p + 1, atom_vir);
  launch_halo_bond_final(e->st, g.B_own, g.B_loc, g.b_src_gid.p, g.b_dst.p, g.b_vec.p, g.gid.p, e->gdb.p, e->gbvec.p,
                         e->forces.p, e->scal.p + 1, atom_vir);
}

// peratom (needs grads): also the per-atom energies and virials of this partition's owned rows and edges
static void run(b2m_engine* e, bool grads, bool peratom = false) {
  B2M_REQUIRE(e->finalized, B2M_ERR_STATE, "weights not finalized");
  B2M_REQUIRE(e->have_graph, B2M_ERR_STATE, "b2m_set_structure has not been called");
  B2M_REQUIRE(e->world == 1 || e->comm != nullptr || e->leader != nullptr || e->debug_no_halo, B2M_ERR_STATE,
              "world > 1 without a communicator (b2m_set_partition is a graph-only view)");
  e->hpoint = 0;
  for (auto& p : e->gather_ev) {
    cudaEventDestroy(p.first);
    cudaEventDestroy(p.second);
  }
  e->gather_ev.clear();
  const long long l0 = g_launch_count;
  B2M_CK(cudaEventRecord(e->ev[0], e->st));
  e->want_grads = grads;
  e->want_peratom = peratom;
  const size_t N = (size_t)e->g.N;
  if (peratom) {
    B2M_REQUIRE(grads, B2M_ERR_INVALID, "per-atom virials need the backward pass");
    e->atom_vir.ensure(N * kAtomVirW), e->atom_e.ensure(N);
    e->atom_vir.zero(N * kAtomVirW, e->st), e->atom_e.zero(N, e->st);
  }
  if (e->kind == 1) tn_forward(e); else forward(e);
  B2M_CK(cudaEventRecord(e->ev[1], e->st));
  if (grads) {
    if (e->kind == 1) tn_backward(e); else backward(e);
  }
  if (peratom)
    launch_atom_energy(e->st, e->g.n_own, e->kind == 1 ? e->tn->e_atom.p : e->e_atom.p, e->g.gid.p, e->g.type.p,
                       e->d_eref, (float)e->desc.data_std, e->desc.data_mean / (double)N, e->atom_e.p);
  if (e->world > 1 && e->leader == nullptr && !e->debug_no_halo) {
    NCCL_CK(g_nccl.AllReduce(e->scal.p, e->scal.p, 10, ncclFloat64, ncclSum, e->comm, e->st));
    if (grads)
      NCCL_CK(g_nccl.AllReduce(e->forces.p, e->forces.p, (size_t)e->g.N * 3, ncclFloat32, ncclSum, e->comm, e->st));
    if (peratom) {
      NCCL_CK(g_nccl.AllReduce(e->atom_vir.p, e->atom_vir.p, N * kAtomVirW, ncclFloat32, ncclSum, e->comm, e->st));
      NCCL_CK(g_nccl.AllReduce(e->atom_e.p, e->atom_e.p, N, ncclFloat64, ncclSum, e->comm, e->st));
    }
  }
  B2M_CK(cudaEventRecord(e->ev[2], e->st));
  B2M_CK(cudaStreamSynchronize(e->st));
  e->launches_last = g_launch_count - l0;
  float ms;
  B2M_CK(cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]));
  e->t_fwd = ms;
  B2M_CK(cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]));
  e->t_bwd = ms;
  double tg = 0;
  for (auto& p : e->gather_ev) {
    B2M_CK(cudaEventElapsedTime(&ms, p.first, p.second));
    tg += ms;
  }
  e->t_gather = e->gather_ev.empty() ? 0 : tg / e->gather_ev.size();
  e->t_total = e->t_fwd + e->t_bwd;
}

// parallel host copy (page-locked <-> pageable): a handful of threads saturate the host memory system, one does not
static void par_memcpy(void* dst, const void* src, size_t bytes) {
  const size_t kMin = 4u << 20;
  unsigned nt = (unsigned)std::min<size_t>(4, bytes / kMin);
  if (nt <= 1) {
    memcpy(dst, src, bytes);
    return;
  }
  std::vector<std::thread> th;
  const size_t chunk = (bytes / nt + 4095) & ~(size_t)4095;
  for (unsigned t = 0; t < nt; t++) {
    const size_t o = (size_t)t * chunk;
    if (o >= bytes) break;
    const size_t n = std::min(chunk, bytes - o);
    th.emplace_back([=] { memcpy((char*)dst + o, (const char*)src + o, n); });
  }
  for (auto& x : th) x.join();
}
static void ensure_pinned(void*& p, size_t& cap, size_t bytes) {
  if (bytes <= cap) return;
  if (p) cudaFreeHost(p);
  p = nullptr, cap = 0;
  B2M_CK(cudaHostAlloc(&p, bytes + bytes / 8, cudaHostAllocDefault));
  cap = bytes + bytes / 8;
}

template <class T>
__global__ void k_add_inplace(int64_t n, const T* __restrict__ src, T* __restrict__ dst) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

// Runs fn(partition) for every partition of a group, one host thread each (each sets its own device); the first
// exception wins and releases the others from the rendezvous.
template <class F>
static void for_each_part(b2m_engine* L, F fn) {
  const int n = (int)L->parts.size();
  L->gsync.reset(n);
  std::vector<std::string> errs(n);
  std::vector<int> codes(n, 0);
  std::vector<std::thread> th;
  for (int p = 0; p < n; p++)
    th.emplace_back([&, p] {
      try {
        B2M_CK(cudaSetDevice(L->parts[p]->device));
        fn(L->parts[p]);
      } catch (const b2m::Error& ex) {
        codes[p] = ex.code, errs[p] = ex.what();
        L->gsync.abort();
      } catch (const std::exception& ex) {
        codes[p] = B2M_ERR_INVALID, errs[p] = ex.what();
        L->gsync.abort();
      }
    });
  for (auto& t : th) t.join();
  cudaSetDevice(L->device);
  for (int p = 0; p < n; p++)
    if (codes[p] != 0 && errs[p].find("a partition of the group failed") == std::string::npos)
      throw Error(codes[p], "partition " + std::to_string(p) + ": " + errs[p]);
  for (int p = 0; p < n; p++)
    if (codes[p] != 0) throw Error(codes[p], errs[p]);
}

static void run_any(b2m_engine* e, bool grads, bool peratom = false) {
  if (e->parts.empty()) {
    run(e, grads, peratom);
    return;
  }
  for_each_part(e, [&](b2m_engine* pe) { run(pe, grads, peratom); });
  // slowest partition = the group's device time; launches summed
  long long launches = 0;
  for (auto* pe : e->parts) {
    e->t_fwd = std::max(e->t_fwd, pe->t_fwd), e->t_bwd = std::max(e->t_bwd, pe->t_bwd);
    e->t_total = std::max(e->t_total, pe->t_total);
    launches += pe->launches_last;
  }
  e->launches_last = launches;
}

static void fetch(b2m_engine* e, double* energy, float* forces, float* stress9) {
  double hs[10];
  B2M_CK(cudaMemcpyAsync(hs, e->scal.p, 10 * sizeof(double), cudaMemcpyDeviceToHost, e->st));
  if (!e->parts.empty() && forces) {  // group: sum the partitions' force arrays on the leader's device
    const size_t n = (size_t)e->g.N * 3;
    e->ftmp.ensure(n + 64);
    for (size_t p = 1; p < e->parts.size(); p++) {
      B2M_CK(cudaMemcpyAsync(e->ftmp.p, e->parts[p]->forces.p, n * sizeof(float), cudaMemcpyDefault, e->st));
      k_add_inplace<<<cdiv((int64_t)n, 256), 256, 0, e->st>>>((int64_t)n, e->ftmp.p, e->forces.p);
      B2M_CK(cudaGetLastError());
    }
  }
  const size_t fbytes = (size_t)e->g.N * 3 * sizeof(float);
  if (forces) {
    ensure_pinned(e->pin_out, e->pin_out_cap, fbytes);
    B2M_CK(cudaMemcpyAsync(e->pin_out, e->forces.p, fbytes, cudaMemcpyDeviceToHost, e->st));
  }
  B2M_CK(cudaStreamSynchronize(e->st));
  if (forces) par_memcpy(forces, e->pin_out, fbytes);
  for (size_t p = 1; p < e->parts.size(); p++) {  // energy and virial of the other partitions
    double ps[10];
    b2m_engine* pe = e->parts[p];
    B2M_CK(cudaSetDevice(pe->device));
    B2M_CK(cudaMemcpy(ps, pe->scal.p, 10 * sizeof(double), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 10; k++) hs[k] += ps[k];
  }
  if (!e->parts.empty()) B2M_CK(cudaSetDevice(e->device));
  e->last_energy = hs[0] + e->desc.data_mean;
  if (energy) *energy = e->last_energy;
  if (stress9)
    for (int k = 0; k < 9; k++) stress9[k] = (float)(hs[1 + k] / e->g.volume * 160.21766208);  // pes.py:140-145
}

// after fetch of a per-atom run: e_i [N] (eV) and W_i [N][9] (eV), global order
static void fetch_peratom(b2m_engine* e, double* atom_energy, float* atom_virial9) {
  const size_t n = (size_t)e->g.N, nw = n * kAtomVirW;
  for (size_t p = 1; p < e->parts.size(); p++) {  // group: sum the partitions' arrays on the leader's device, as fetch
    b2m_engine* pe = e->parts[p];                  // does the forces
    e->avtmp.ensure(nw), e->aetmp.ensure(n);
    B2M_CK(cudaMemcpyAsync(e->avtmp.p, pe->atom_vir.p, nw * sizeof(float), cudaMemcpyDefault, e->st));
    k_add_inplace<<<cdiv((int64_t)nw, 256), 256, 0, e->st>>>((int64_t)nw, e->avtmp.p, e->atom_vir.p);
    B2M_CK(cudaGetLastError());
    B2M_CK(cudaMemcpyAsync(e->aetmp.p, pe->atom_e.p, n * sizeof(double), cudaMemcpyDefault, e->st));
    k_add_inplace<<<cdiv((int64_t)n, 256), 256, 0, e->st>>>((int64_t)n, e->aetmp.p, e->atom_e.p);
    B2M_CK(cudaGetLastError());
  }
  std::vector<float> rows(atom_virial9 ? nw : 0);
  if (atom_energy) B2M_CK(cudaMemcpyAsync(atom_energy, e->atom_e.p, n * sizeof(double), cudaMemcpyDeviceToHost, e->st));
  if (atom_virial9)
    B2M_CK(cudaMemcpyAsync(rows.data(), e->atom_vir.p, nw * sizeof(float), cudaMemcpyDeviceToHost, e->st));
  B2M_CK(cudaStreamSynchronize(e->st));
  if (atom_virial9)
    for (size_t i = 0; i < n; i++) memcpy(atom_virial9 + i * 9, rows.data() + i * kAtomVirW, 9 * sizeof(float));
}

}  // namespace b2m

// ==========================================================================================
// C ABI
// ==========================================================================================
#define API_BEGIN                               \
  if (!h) return B2M_ERR_INVALID;               \
  try {                                         \
    cudaSetDevice(h->device);
#define API_END                                 \
  }                                             \
  catch (const b2m::Error& ex) {                \
    h->err = ex.what();                         \
    return ex.code;                             \
  }                                             \
  catch (const std::exception& ex) {            \
    h->err = ex.what();                         \
    return B2M_ERR_INVALID;                     \
  }                                             \
  return B2M_OK;

static std::string g_create_err;

// partition of a single-process group that the inspection calls address (b2m_set_view; the handle itself otherwise)
static b2m_engine* viewed(b2m_engine* h) { return h->parts.empty() ? h : h->parts[h->view]; }

// every partition of a single-process group holds the replicated weights (chgnet.py:455-549 deep-copies them per GPU)
template <class F>
static void each_member(b2m_engine* h, F fn) {
  if (h->parts.empty()) {
    fn(h);
    return;
  }
  for (auto* pe : h->parts) {
    B2M_CK(cudaSetDevice(pe->device));
    fn(pe);
  }
  B2M_CK(cudaSetDevice(h->device));
}


extern "C" {

static b2m_engine* create_one(const b2m_model_desc* desc, int device, int count) {
  B2M_REQUIRE(device >= 0 && device < count, B2M_ERR_INVALID, "bad device ordinal");
  b2m_engine* e = new b2m_engine();
  try {
    e->desc = *desc;
    e->device = device;
    B2M_CK(cudaSetDevice(e->device));
    cudaDeviceProp prop;
    B2M_CK(cudaGetDeviceProperties(&prop, e->device));
    if (prop.major != 10) throw Error(B2M_ERR_CUDA, "libb200mlip is built for sm_100a (B200) only");
    e->num_sms = prop.multiProcessorCount;
    const char* leg = getenv("B2M_LEGACY_FFMA");
    e->use_tc = !(leg && leg[0] == '1');
    const char* gen = getenv("B2M_ATOMCONV");
    e->ac_gen = gen ? atoi(gen) : 3;
    const char* nh = getenv("B2M_DEBUG_NO_HALO");
    e->debug_no_halo = nh && nh[0] == '1';
    B2M_CK(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking));
    B2M_CK(cudaStreamCreateWithFlags(&e->cst, cudaStreamNonBlocking));
    B2M_CK(cudaEventCreateWithFlags(&e->ev_prod, cudaEventDisableTiming));
    B2M_CK(cudaEventCreateWithFlags(&e->ev_halo, cudaEventDisableTiming));
    for (auto& ev : e->ev) B2M_CK(cudaEventCreate(&ev));
  } catch (...) {
    delete e;
    throw;
  }
  return e;
}

static int create_any(const b2m_model_desc* desc, const b2m_tensornet_desc* tdesc, const int* devices, int ndev,
                      b2m_handle* out) {
  if (!desc || !devices || !out) return B2M_ERR_INVALID;
  std::vector<b2m_engine*> made;
  try {
    B2M_REQUIRE(ndev >= 1 && ndev <= MAXP, B2M_ERR_PARTITIONS, "ndev must be in [1,16]");
    if (tdesc) {
      B2M_REQUIRE(tdesc->units == D, B2M_ERR_INVALID, "TensorNet engine supports units = 64");
      B2M_REQUIRE(tdesc->num_rbf >= 1 && tdesc->num_rbf <= 64, B2M_ERR_INVALID, "num_rbf must be in [1,64]");
      B2M_REQUIRE(tdesc->n_blocks >= 1 && tdesc->n_blocks <= 16, B2M_ERR_INVALID, "nblocks must be in [1,16]");
      B2M_REQUIRE(tdesc->cutoff > 0 && tdesc->rbf_width > 0, B2M_ERR_INVALID, "cutoff and rbf width must be positive");
    } else {
      B2M_REQUIRE(desc->dim == D && desc->max_n == NR && desc->max_f == 4, B2M_ERR_INVALID,
                  "engine supports dim=64, max_n=9, max_f=4");
      B2M_REQUIRE(desc->n_blocks >= 2 && desc->n_blocks <= 16, B2M_ERR_INVALID, "n_blocks must be in [2,16]");
      B2M_REQUIRE(desc->cutoff > 0 && desc->three_body_cutoff > 0 && desc->three_body_cutoff <= desc->cutoff,
                  B2M_ERR_INVALID, "bond_r cannot be greater than regular cutoff");
    }
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count <= 0)
      throw Error(B2M_ERR_CUDA, std::string("no CUDA device available (libb200mlip has no CPU fallback): ") +
                                    cudaGetErrorString(ce));
    for (int p = 0; p < ndev; p++) {
      made.push_back(create_one(desc, devices[p], count));
      if (tdesc) {
        b2m_engine* m = made.back();
        m->kind = 1;
        m->tn = new TnState();
        m->tn->units = tdesc->units, m->tn->num_rbf = tdesc->num_rbf, m->tn->nblocks = tdesc->n_blocks;
        m->tn->so3 = tdesc->so3 ? 1 : 0;
        m->tn->rp.nr = tdesc->num_rbf, m->tn->rp.nrp = 64;
        m->tn->rp.width = (float)tdesc->rbf_width, m->tn->rp.rc = (float)tdesc->cutoff;
        for (float& v : m->tn->rp.mu) v = 0.f;
      }
    }
    b2m_engine* e = made[0];
    if (ndev > 1) {
      // single-process group: partition p lives on devices[p] (ordinals may repeat: several partitions on one GPU);
      // peer access between distinct devices so that halo rows are plain stores into the neighbour's memory
      for (int p = 0; p < ndev; p++) {
        made[p]->rank = p, made[p]->world = ndev, made[p]->leader = e;
        B2M_CK(cudaSetDevice(made[p]->device));
        made[p]->hev.resize(4 * 16 + 8);  // 2 forward + 2 backward exchange points per block, n_blocks <= 16
        for (auto& ev : made[p]->hev) B2M_CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        for (int q = 0; q < ndev; q++) {
          if (made[q]->device == made[p]->device) continue;
          int can = 0;
          B2M_CK(cudaDeviceCanAccessPeer(&can, made[p]->device, made[q]->device));
          B2M_REQUIRE(can, B2M_ERR_CUDA, "devices of a single-process group need peer access (NVLink / NVSwitch)");
          cudaError_t pe = cudaDeviceEnablePeerAccess(made[q]->device, 0);
          if (pe == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
          else B2M_CK(pe);
        }
      }
      e->parts = made;
      B2M_CK(cudaSetDevice(e->device));
    }
    *out = e;
  } catch (const b2m::Error& ex) {
    for (auto* m : made) {
      delete m->tn;
      delete m;
    }
    g_create_err = ex.what();
    return ex.code;
  }
  return B2M_OK;
}

int b2m_create(const b2m_model_desc* desc, const int* devices, int ndev, b2m_handle* out) {
  return create_any(desc, nullptr, devices, ndev, out);
}

int b2m_create_tensornet(const b2m_tensornet_desc* tdesc, const int* devices, int ndev, b2m_handle* out) {
  if (!tdesc) return B2M_ERR_INVALID;
  // the shared part of the engine (graph build, scaling, transport) reads the CHGNet-shaped description: no bond graph
  // (use_bond_graph False, three_body_cutoff 0: pes.py:79-80)
  b2m_model_desc d;
  memset(&d, 0, sizeof d);
  d.n_elem = tdesc->n_elem, d.dim = D, d.max_n = NR, d.max_f = 4, d.n_blocks = tdesc->n_blocks, d.cutoff_exponent = 0;
  d.cutoff = tdesc->cutoff, d.three_body_cutoff = 0.0, d.data_mean = tdesc->data_mean, d.data_std = tdesc->data_std;
  return create_any(&d, tdesc, devices, ndev, out);
}

static void destroy_one(b2m_engine* h) {
  cudaSetDevice(h->device);
  delete h->tn;  // frees its device buffers
  if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  for (auto& p : h->gather_ev) {
    cudaEventDestroy(p.first);
    cudaEventDestroy(p.second);
  }
  for (auto& ev : h->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto& ev : h->hev) cudaEventDestroy(ev);
  if (h->pin_in) cudaFreeHost(h->pin_in);
  if (h->pin_out) cudaFreeHost(h->pin_out);
  if (h->ev_prod) cudaEventDestroy(h->ev_prod);
  if (h->ev_halo) cudaEventDestroy(h->ev_halo);
  if (h->cst) cudaStreamDestroy(h->cst);
  if (h->st) cudaStreamDestroy(h->st);
  delete h;
}

int b2m_destroy(b2m_handle h) {
  if (!h) return B2M_ERR_INVALID;
  std::vector<b2m_engine*> members(h->parts.begin(), h->parts.end());
  for (size_t p = 1; p < members.size(); p++) destroy_one(members[p]);
  destroy_one(h);
  return B2M_OK;
}

const char* b2m_last_error(b2m_handle h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int b2m_load_weights(b2m_handle h, const char* name, const float* host_ptr, const int64_t* shape, int ndim) {
  API_BEGIN
  B2M_REQUIRE(name && host_ptr && shape && ndim >= 1 && ndim <= 4, B2M_ERR_INVALID, "bad weight arguments");
  size_t n = 1;
  std::vector<int64_t> sh(shape, shape + ndim);
  for (auto s : sh) n *= (size_t)s;
  each_member(h, [&](b2m_engine* e) {
    e->host_w[name] = std::vector<float>(host_ptr, host_ptr + n);
    e->host_shape[name] = sh;
    e->finalized = false;
  });
  API_END
}

int b2m_set_element_refs(b2m_handle h, const double* offsets, int n) {
  API_BEGIN
  B2M_REQUIRE(offsets == nullptr || n == 0 || n == h->desc.n_elem, B2M_ERR_INVALID, "element_refs length must equal n_elem");
  each_member(h, [&](b2m_engine* e) {
    if (offsets == nullptr || n == 0) {  // clear: a later Potential without element_refs must not inherit the old offsets
      e->elem_refs.clear();
      e->d_eref = nullptr;
    } else {
      e->elem_refs.assign(offsets, offsets + n);
    }
    e->finalized = false;
  });
  API_END
}

int b2m_set_scaling(b2m_handle h, double data_mean, double data_std) {
  API_BEGIN
  each_member(h, [&](b2m_engine* e) {
    e->desc.data_mean = data_mean;
    e->desc.data_std = data_std;
  });
  API_END
}

int b2m_finalize_weights(b2m_handle h) {
  API_BEGIN
  each_member(h, [&](b2m_engine* e) {
    if (e->kind == 1) tn_finalize_weights(e); else finalize_weights(e);
  });
  API_END
}

int b2m_comm_unique_id(char* out128) {
  if (!out128) return B2M_ERR_INVALID;
  try {
    g_nccl.load();
    ncclUniqueId id;
    NCCL_CK(g_nccl.GetUniqueId(&id));
    static_assert(sizeof(id) == 128, "ncclUniqueId size");
    memcpy(out128, &id, 128);
  } catch (const b2m::Error& ex) {
    g_create_err = ex.what();
    return ex.code;
  }
  return B2M_OK;
}

int b2m_comm_init(b2m_handle h, const char* id128, int rank, int world) {
  API_BEGIN
  B2M_REQUIRE(world >= 1 && world <= MAXP && rank >= 0 && rank < world, B2M_ERR_PARTITIONS, "bad rank/world");
  B2M_REQUIRE(h->parts.empty(), B2M_ERR_STATE, "a single-process group (ndev > 1) needs no communicator");
  h->rank = rank;
  h->world = world;
  if (world > 1) {
    B2M_REQUIRE(id128 != nullptr, B2M_ERR_INVALID, "unique id required");
    g_nccl.load();
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    NCCL_CK(g_nccl.CommInitRank(&h->comm, world, id, rank));
  }
  API_END
}

int b2m_set_partition(b2m_handle h, int rank, int world) {
  API_BEGIN
  B2M_REQUIRE(world >= 1 && world <= MAXP && rank >= 0 && rank < world, B2M_ERR_PARTITIONS, "bad rank/world");
  B2M_REQUIRE(h->comm == nullptr, B2M_ERR_STATE, "communicator already initialised");
  B2M_REQUIRE(h->parts.empty(), B2M_ERR_STATE, "the partitions of a single-process group are fixed by b2m_create");
  h->rank = rank;
  h->world = world;
  h->have_graph = false;
  API_END
}

static void set_structure_one(b2m_engine* h, int64_t natoms, const double* cart, const double* lattice9,
                              const int32_t* species, const int* pbc3, double tol) {
  h->have_graph = false;
  // positions and species through the library's page-locked staging (asynchronous upload inside the build)
  if (natoms > 0 && natoms < (1LL << 31) / 4) {
    const size_t cb = (size_t)natoms * 3 * sizeof(double), sb = (size_t)natoms * sizeof(int32_t);
    ensure_pinned(h->pin_in, h->pin_in_cap, cb + sb);
    par_memcpy(h->pin_in, cart, cb);
    memcpy((char*)h->pin_in + cb, species, sb);
    cart = reinterpret_cast<const double*>(h->pin_in);
    species = reinterpret_cast<const int32_t*>((const char*)h->pin_in + cb);
  }
  B2M_CK(cudaEventRecord(h->ev[3], h->st));
  h->g.build(h->st, natoms, cart, lattice9, species, pbc3, h->desc.cutoff, h->desc.three_body_cutoff, tol, h->rank,
             h->world);
  if (h->kind == 1) tn_alloc_workspace(h); else alloc_workspace(h);
  B2M_CK(cudaEventRecord(h->ev[4], h->st));
  B2M_CK(cudaStreamSynchronize(h->st));
  float ms;
  B2M_CK(cudaEventElapsedTime(&ms, h->ev[3], h->ev[4]));
  h->t_graph = ms;
  h->have_graph = true;
}

int b2m_set_structure(b2m_handle h, int64_t natoms, const double* cart, const double* lattice9,
                      const int32_t* species, const int* pbc3, double tol) {
  API_BEGIN
  B2M_REQUIRE(cart && lattice9 && species && pbc3, B2M_ERR_INVALID, "null structure argument");
  if (h->parts.empty()) {
    set_structure_one(h, natoms, cart, lattice9, species, pbc3, tol);
  } else {  // every partition builds its own slab on its own device, concurrently
    for_each_part(h, [&](b2m_engine* pe) { set_structure_one(pe, natoms, cart, lattice9, species, pbc3, tol); });
    for (auto* pe : h->parts) h->t_graph = std::max(h->t_graph, pe->t_graph);
  }
  API_END
}

int b2m_compute(b2m_handle h, int want_forces, int want_stress, double* energy, float* forces, float* stress9) {
  API_BEGIN
  run_any(h, want_forces || want_stress);
  fetch(h, energy, want_forces ? forces : nullptr, want_stress ? stress9 : nullptr);
  API_END
}

int b2m_compute_peratom(b2m_handle h, int want_forces, double* energy, float* forces, float* stress9,
                        double* atom_energy, float* atom_virial9) {
  API_BEGIN
  run_any(h, true, true);
  fetch(h, energy, want_forces ? forces : nullptr, stress9);
  fetch_peratom(h, atom_energy, atom_virial9);
  API_END
}

int b2m_compute_resident(b2m_handle h, int want_forces, int want_stress, int reps, double* energy, float* ms) {
  API_BEGIN
  B2M_REQUIRE(reps >= 1, B2M_ERR_INVALID, "reps >= 1");
  for (int r = 0; r < reps; r++) run_any(h, want_forces || want_stress);
  fetch(h, energy, nullptr, nullptr);
  if (ms) *ms = (float)h->t_total;
  API_END
}

int b2m_get_sitewise(b2m_handle h, float* out) {
  API_BEGIN
  B2M_REQUIRE(h->have_graph && out, B2M_ERR_STATE, "no structure");
  B2M_REQUIRE(h->kind == 0, B2M_ERR_INVALID, "the site-wise readout belongs to CHGNet (TensorNet has none)");
  std::vector<float> full(h->g.N, 0.f);
  auto collect = [&](b2m_engine* e) {  // owned rows of one partition -> global order
    Graph& g = e->g;
    std::vector<float> loc(g.n_own);
    std::vector<int> gid(g.n_own);
    B2M_CK(cudaMemcpyAsync(loc.data(), e->site.p, g.n_own * sizeof(float), cudaMemcpyDeviceToHost, e->st));
    B2M_CK(cudaMemcpyAsync(gid.data(), g.gid.p, g.n_own * sizeof(int), cudaMemcpyDeviceToHost, e->st));
    B2M_CK(cudaStreamSynchronize(e->st));
    for (int i = 0; i < g.n_own; i++) full[gid[i]] = loc[i];
  };
  each_member(h, collect);
  Graph& g = h->g;
  if (h->world > 1 && h->parts.empty()) {
    B2M_CK(cudaMemcpyAsync(h->site_full.p, full.data(), g.N * sizeof(float), cudaMemcpyHostToDevice, h->st));
    NCCL_CK(g_nccl.AllReduce(h->site_full.p, h->site_full.p, (size_t)g.N, ncclFloat32, ncclSum, h->comm, h->st));
    B2M_CK(cudaMemcpyAsync(full.data(), h->site_full.p, g.N * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    B2M_CK(cudaStreamSynchronize(h->st));
  }
  memcpy(out, full.data(), g.N * sizeof(float));
  API_END
}

int b2m_set_view(b2m_handle h, int part) {
  API_BEGIN
  const int n = h->parts.empty() ? 1 : (int)h->parts.size();
  B2M_REQUIRE(part >= 0 && part < n, B2M_ERR_PARTITIONS, "no such partition in this handle");
  h->view = part;
  API_END
}

int b2m_get_counts(b2m_handle h, int64_t* out, int n) {
  API_BEGIN
  B2M_REQUIRE(out && n >= 10, B2M_ERR_INVALID, "need room for 10 counts");
  b2m_engine* v = viewed(h);
  Graph& g = v->g;
  out[0] = g.n_own, out[1] = g.n_halo, out[2] = g.E, out[3] = g.B_own, out[4] = g.B_halo, out[5] = g.A;
  out[6] = g.axis, out[7] = v->rank, out[8] = v->world, out[9] = h->launches_last;
  API_END
}

int64_t b2m_get_partition_info(b2m_handle h, int which, int64_t* out, int64_t cap) {
  if (!h) return B2M_ERR_INVALID;
  try {
    b2m_engine* v = viewed(h);
    cudaSetDevice(v->device);
    B2M_REQUIRE(v->have_graph && out, B2M_ERR_STATE, "no structure");
    const int64_t n = v->g.export_info(v->st, which, out, cap);
    cudaSetDevice(h->device);
    return n;
  } catch (const b2m::Error& ex) {
    h->err = ex.what();
    return ex.code;
  }
}

int b2m_debug_tensor(b2m_handle h, const char* name, float* out, int64_t cap, int64_t* rows, int64_t* cols) {
  API_BEGIN
  B2M_REQUIRE(h->have_graph && name && out && rows && cols, B2M_ERR_STATE, "no structure");
  Graph& g = h->g;
  std::string n(name);
  const float* src = nullptr;
  int64_t r = 0, c = D;
  auto idx = [&](const std::string& pre) { return atoi(n.c_str() + pre.size()); };
  if (h->kind == 1) {
    B2M_REQUIRE(tn_debug_lookup(h, n, src, r, c), B2M_ERR_INVALID, "unknown debug tensor: " + n);
  } else if (n[0] == 'x' && isdigit(n[1])) {
    int l = idx("x");
    B2M_REQUIRE(l >= 0 && l < (int)h->x.size(), B2M_ERR_INVALID, "bad layer");
    src = h->x[l].p, r = l == (int)h->x.size() - 1 ? g.n_own : g.n_loc;
  } else if (n[0] == 'h' && isdigit(n[1])) {
    int l = idx("h");
    B2M_REQUIRE(l >= 0 && l < (int)h->h.size(), B2M_ERR_INVALID, "bad layer");
    src = h->h[l].p, r = g.B_own;
  } else if (n.rfind("ang", 0) == 0 && isdigit(n[3])) {
    int l = idx("ang");
    B2M_REQUIRE(l >= 0 && l < (int)h->ang.size(), B2M_ERR_INVALID, "bad layer");
    src = h->ang[l].p, r = g.A;
  } else if (n == "e_atom") {
    src = h->e_atom.p, r = g.n_own, c = 1;
  } else if (n == "gd") {
    src = h->gd.p, r = g.E, c = 1;
  } else if (n == "gdb") {
    src = h->gdb.p, r = g.B_loc, c = 1;
  } else if (n == "gbvec") {
    src = h->gbvec.p, r = g.B_loc, c = 3;
  } else if (n == "gx") {
    src = h->gx.p, r = g.n_loc;
  } else if (n == "gh") {
    src = h->gh.p, r = g.B_loc;
  } else if (n == "gang") {
    src = h->gang.p, r = g.A;
  } else if (n == "e_vec") {
    src = reinterpret_cast<const float*>(g.e_vec.p), r = g.E, c = 4;
  } else {
    throw Error(B2M_ERR_INVALID, "unknown debug tensor: " + n);
  }
  B2M_REQUIRE(r * c <= cap, B2M_ERR_INVALID, "debug buffer too small");
  const bool angle_tensor = n.rfind("ang", 0) == 0 || n == "gang";
  if (angle_tensor && h->use_tc) {  // tile-interleaved on the device: hand the caller the logical [A][64] rows
    const size_t padded = (size_t)(r + 127) / 128 * 128 * 64;
    std::vector<float> tmp(padded);
    B2M_CK(cudaMemcpyAsync(tmp.data(), src, padded * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    B2M_CK(cudaStreamSynchronize(h->st));
    for (int64_t i = 0; i < r; i++)
      for (int k = 0; k < 64; k++) out[i * 64 + k] = tmp[ang_index(i, k, 1)];
  } else {
    B2M_CK(cudaMemcpyAsync(out, src, r * c * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    B2M_CK(cudaStreamSynchronize(h->st));
  }
  *rows = r, *cols = c;
  API_END
}

int b2m_release_workspace(b2m_handle h) {
  API_BEGIN
  each_member(h, [&](b2m_engine* e) {
    B2M_CK(cudaStreamSynchronize(e->st));
    e->have_graph = false;
    auto drop = [](auto& b) {
      if (b.p) cudaFree(b.p);
      b.p = nullptr, b.cap = 0;
    };
    for (auto* v : {&e->x, &e->h, &e->ang, &e->upd, &e->uv, &e->uvB, &e->dsB, &e->uvA, &e->ApL, &e->CpL, &e->QpL})
      for (auto& b : *v) drop(b);
    for (auto* b : {&e->be_e, &e->dbe_e, &e->Ha, &e->Hb, &e->Xc, &e->agg, &e->aggB, &e->y1p, &e->y1, &e->y2p, &e->y2,
                    &e->e_atom, &e->site, &e->gx, &e->gh, &e->gang, &e->gA, &e->gC, &e->gQ, &e->gHa, &e->gHb, &e->gXc,
                    &e->gagg, &e->gupd, &e->gaggB, &e->gd, &e->gdb, &e->gbvec, &e->gy1, &e->gy2, &e->forces,
                    &e->sendbuf, &e->recvbuf, &e->site_full, &e->precv[0], &e->precv[1], &e->ftmp, &e->atom_vir,
                    &e->avtmp})
      drop(*b);
    drop(e->atom_e), drop(e->aetmp);
    tn_release(e);
    e->g.~Graph();  // the resident graph goes too
    new (&e->g) Graph();
  });
  API_END
}

int b2m_last_timings(b2m_handle h, double* out, int n) {
  API_BEGIN
  B2M_REQUIRE(out && n >= 5, B2M_ERR_INVALID, "need room for 5 timings");
  out[0] = h->t_graph, out[1] = h->t_fwd, out[2] = h->t_bwd, out[3] = h->t_gather, out[4] = h->t_total;
  API_END
}

}  // extern "C"
