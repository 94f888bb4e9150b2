// rbt_api.cu -- C ABI of librobotoc_b200.so (see include/robotoc_b200.h for the reference interfaces replaced).
// Plumbing only: handles, device buffers, stream-ordered copies and kernel launches.  No CPU compute path.
#include <cstdio>
#include <cstring>
#include <cstdint>
#include <cstdlib>
#include <memory>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>

#include "../../include/robotoc_b200.h"
#include "riccati_backward.cuh"
#include "riccati_forward.cuh"
#include "riccati_unconstr.cuh"
#include "stage_kernels.cuh"
#include "ustage_kernels.cuh"
#include "eval_kernels.cuh"
#include "line_search_kernels.cuh"

namespace {

struct Err {
  std::string msg;
};

#define RBT_CUDA(h, call)                                                                     \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                          \
      return RBT_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

// Device memory, streams and events owned by a handle: released when the handle is deleted (after rbt_destroy has made
// the handle's device current).
struct CudaRelease {
  void operator()(void* p) const { cudaFree(p); }
  void operator()(CUstream_st* s) const { cudaStreamDestroy(s); }
  void operator()(CUevent_st* e) const { cudaEventDestroy(e); }
};
template <class T>
using Owned = std::unique_ptr<T, CudaRelease>;

template <class T>
cudaError_t dev_alloc(Owned<T>& p, size_t n) {
  p.reset();
  T* q = nullptr;
  const cudaError_t e = cudaMalloc(&q, n * sizeof(T));
  p.reset(q);
  return e;
}

// The public buffers of a handle, indexed by RBT_BUF_*.  `ptr` is what the kernels use: the handle's own allocation, or
// a caller's buffer bound with rbt_bind_buffer (never freed by the handle).
struct BufTable {
  struct Entry {
    Owned<double> own;
    double* ptr = nullptr;
    int per_row = 0;        // doubles per row
    bool per_grid = false;  // a row per grid point of every OCP (else one row per OCP)
  };
  Entry e[RBT_BUF_PERF + 1];
  long long batch = 0;
  int n_grid_max = 0;

  static bool valid(int which) { return which >= 0 && which <= RBT_BUF_PERF; }
  double* operator[](int which) const { return valid(which) ? e[which].ptr : nullptr; }
  long long doubles(int which, int n_grid) const {
    if (!valid(which) || !e[which].own) return -1;
    return batch * (e[which].per_grid ? n_grid : 1) * e[which].per_row;
  }
  // the handle's own allocation, zeroed
  cudaError_t alloc(int which, int per_row, bool per_grid) {
    Entry& x = e[which];
    x.per_row = per_row;
    x.per_grid = per_grid;
    const size_t n = size_t(batch) * (per_grid ? n_grid_max : 1) * per_row;
    const cudaError_t err = dev_alloc(x.own, n);
    x.ptr = x.own.get();
    return err != cudaSuccess ? err : cudaMemset(x.ptr, 0, n * 8);
  }
};

// A contiguous range [b0, b0 + nb) of the batch that a launch or a copy works on.
struct Win {
  int b0, nb;
};

}  // namespace

struct rbt_handle {
  rbt_dims dims;
  rbt_layout L;
  int n_grid_max = 0, n_grid = 0, batch = 0, device = 0;
  double max_dts0 = 0.1;
  Owned<rbt_stage_ctrl> d_ctrl;
  std::vector<rbt_stage_ctrl> ctrl;  // host copy
  BufTable buf;
  Owned<int> d_info;
  Owned<int> d_struct;  // [0]: 1 = every Fxx of the KKT buffer has the mechanical structure (see rbt_set_fxx_structure)
  int fxx_mode = RBT_FXX_AUTO;
  bool kkt_from_condense = false;  // the KKT records were just written by rbt_condense: structure holds by construction
  // stage layer
  bool stage_ready = false;
  bool keep_info = false;  // condense's Cholesky flags survive the following backward launch
  rbt_stage_dims sdims;
  rbt_stage_layout S;
  rbt_constraint_table table;
  Owned<double> d_ones, d_stage_perf, d_x0in;  // eval_kernels.cuh
  // line search (line_search_kernels.cuh): trial buffers sized on first use, filter state per OCP
  int ls_trials = 0;
  Owned<double> d_ls_alphas, d_ls_trial, d_ls_stage_barrier, d_ls_barrier, d_ls_in, d_ls_filt, d_ls_step;
  Owned<int> d_ls_nfilt, d_ls_k;
  Owned<double> d_step_pack;  // packed Newton step of this rank (rbt_allgather_step), allocated on first use
  long long launches = 0;
  Owned<double> d_wire;       // packed host wire records (rbt_iteration_host_wire), allocated on first use
  Owned<int> d_tgt;           // box rows per PDIPM target (stage_kernels.cuh: StageParams::tgt)
  Owned<double> d_bound;      // joint limits per box row (rbt_set_joint_limits)
  Owned<double> d_res_stage;  // rbt_iteration_host_resident: compact residuals in, compact slack|dual out
  Owned<double> d_sd_stage;
  std::vector<rbt_wire_layout> Wv;   // per grid point (the wire record of a grid point depends on its control word)
  Owned<rbt_wire_layout> d_W;
  long long w_ocp = 0;               // doubles of one OCP's concatenated wire records
  int cost_structure = RBT_COST_GENERAL;  // what the host's wire records hold (rbt_set_wire_cost_structure)
  bool wire_dirty = true;                 // per-grid-point wire layouts on the device are stale (schedule / cost structure changed)
  bool attr_bwd = false, attr_fwd = false, attr_cond = false;  // MaxDynamicSharedMemorySize set on THIS handle's device
  cudaEvent_t ev_condense_mid = nullptr;  // caller-owned event recorded between the two kernels of rbt_condense (timing)
  Owned<CUstream_st> s_h2d, s_d2h;
  std::vector<Owned<CUevent_st>> ev;
  std::string err;
};

struct rbt_uhandle {
  int nv = 0, N = 0, batch = 0, device = 0;
  double dt = 0;
  rbt_ulayout L;
  BufTable buf;
  Owned<int> d_info;
  // stage layer
  bool stage_ready = false;
  rbt_ustage_layout S;
  rbt_constraint_table table;
  Owned<double> d_ones;
  long long launches = 0;
  std::string err;
};

// ---- compiled instances ------------------------------------------------------------------------------------------
// constrained: ANYmal (floating base + 4 point contacts), nv=18, nu=12, max_dimf=12     src/robot/robot.cpp:33-60
constexpr int INST_NV = 18, INST_NU = 12, INST_NS = 12;
// unconstrained: iiwa14, nv=7
constexpr int UINST_NV = 7;

// All functions below are declared extern "C" in include/robotoc_b200.h; the definitions inherit that linkage.

const char* rbt_version(void) { return "robotoc_b200 0.1 (sm_100a; instances: constrained nv18/nu12/ns12; unconstr nv7)"; }

int rbt_layout_get(const rbt_dims* dims, const char* field) {
  if (!dims || !field) return -1;
  rbt_layout L;
  rbt_make_layout(dims, &L);
  return rbt_layout_field(&L, field);
}

int rbt_ulayout_get(int nv, const char* field) {
  if (nv <= 0 || !field) return -1;
  rbt_ulayout L;
  rbt_make_ulayout(nv, &L);
  return rbt_ulayout_field(&L, field);
}

int rbt_device_info(int device, int* sm, int* n_sm, char* name, int name_len) {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    cudaGetLastError();
    return RBT_ERR_CUDA;
  }
  if (sm) *sm = prop.major * 10 + prop.minor;
  if (n_sm) *n_sm = prop.multiProcessorCount;
  if (name && name_len > 0) {
    std::strncpy(name, prop.name, name_len - 1);
    name[name_len - 1] = 0;
  }
  return RBT_OK;
}

int rbt_create(const rbt_dims* dims, int n_grid_max, int batch, int device, rbt_handle** out) {
  if (!dims || !out || n_grid_max < 2 || batch < 1 || dims->nv < 1 || dims->nu < 1 || dims->ns_max < 0) return RBT_ERR_ARG;
  if (dims->nv != INST_NV || dims->nu != INST_NU || dims->ns_max != INST_NS) return RBT_ERR_ARG;
  rbt_handle* h = new rbt_handle();
  h->dims = *dims;
  rbt_make_layout(dims, &h->L);
  h->n_grid_max = n_grid_max;
  h->batch = batch;
  h->device = device;
  h->buf.batch = batch;
  h->buf.n_grid_max = n_grid_max;
  *out = h;
  RBT_CUDA(h, cudaSetDevice(device));
  RBT_CUDA(h, dev_alloc(h->d_ctrl, n_grid_max));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_KKT, h->L.k_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_RIC, h->L.r_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_FACT, h->L.f_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_DIR, h->L.d_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_DX0, h->L.nx, false));
  RBT_CUDA(h, dev_alloc(h->d_info, batch));
  RBT_CUDA(h, dev_alloc(h->d_struct, 4));
  RBT_CUDA(h, cudaMemset(h->d_struct.get(), 0, 4 * sizeof(int)));
  RBT_CUDA(h, cudaMemset(h->d_info.get(), 0, size_t(batch) * sizeof(int)));
  return RBT_OK;
}

// The stage kernels are compiled for nf_max / n_contacts of the constraint table: every grid of the schedule must fit.
static int check_contacts(rbt_handle* h, const rbt_stage_ctrl* ctrl, int n_grid) {
  if (!h->stage_ready) return RBT_OK;
  for (int i = 0; i < n_grid; ++i)
    if (ctrl[i].nf > h->sdims.nf_max || ctrl[i].contact_mask >= (1 << h->sdims.n_contacts)) {
      h->err = "[rbt_set_schedule] invalid argument: grid " + std::to_string(i) + " has more contacts than the stage layer was set up for";
      return RBT_ERR_ARG;
    }
  return RBT_OK;
}

int rbt_destroy(rbt_handle* h) {
  if (!h) return RBT_ERR_ARG;
  cudaSetDevice(h->device);
  delete h;
  return RBT_OK;
}

int rbt_set_schedule(rbt_handle* h, const rbt_stage_ctrl* ctrl, int n_grid, double max_dts0) {
  if (!h || !ctrl) return RBT_ERR_ARG;
  if (n_grid < 2 || n_grid > h->n_grid_max) {
    h->err = "[rbt_set_schedule] invalid argument: n_grid must be in [2, n_grid_max]";
    return RBT_ERR_ARG;
  }
  if (!(max_dts0 > 0)) {
    h->err = "[rbt_set_schedule] invalid argument: max_dts0 must be positive";
    return RBT_ERR_ARG;
  }
  for (int i = 0; i < n_grid; ++i) {
    const rbt_stage_ctrl& c = ctrl[i];
    const bool last = (i == n_grid - 1);
    if ((c.type == RBT_TERMINAL) != last || c.type < 0 || c.type > 3 || c.ns < 0 || c.ns > h->dims.ns_max ||
        (c.type == RBT_IMPACT && (i == 0 || last)) || (c.type == RBT_LIFT && i == 0)) {
      h->err = "[rbt_set_schedule] invalid argument: inconsistent stage control table at grid " + std::to_string(i);
      return RBT_ERR_ARG;
    }
    // contact bookkeeping: the stage kernels index fixed-size shared arrays with nv + nf and use popc(contact_mask) offsets
    // into the stacked force block, so a table that lies about either is rejected here, not discovered on the device
    const int nf_max = 3 * RBT_MAX_CONTACTS;
    if (c.nf < 0 || c.nf > nf_max || c.nf % 3 != 0 || c.contact_mask < 0 || c.contact_mask >= (1 << RBT_MAX_CONTACTS) ||
        3 * __builtin_popcount((unsigned)c.contact_mask) != c.nf || c.ngrids_in_phase < 0 || !(c.dt >= 0.0) ||
        !(c.dt < 1.0e300) || (c.sto != 0 && c.sto != 1) || (c.sto_next != 0 && c.sto_next != 1) || c.ineq_gate < 0 ||
        c.ineq_gate > 2) {
      h->err = "[rbt_set_schedule] invalid argument: grid " + std::to_string(i) +
               ": need 0 <= nf <= 12, nf % 3 == 0, 3 * popcount(contact_mask) == nf, ngrids_in_phase >= 0, finite dt >= 0, "
               "ineq_gate in {0, 1, 2}";
      return RBT_ERR_ARG;
    }
    if (c.type == RBT_IMPACT && c.ns != 0) {
      h->err = "[rbt_set_schedule] invalid argument: an impact grid carries no switching constraint (grid " + std::to_string(i) + ")";
      return RBT_ERR_ARG;
    }
  }
  if (check_contacts(h, ctrl, n_grid) != RBT_OK) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaMemcpy(h->d_ctrl.get(), ctrl, sizeof(rbt_stage_ctrl) * n_grid, cudaMemcpyHostToDevice));
  // stage-conditional outputs (M, STO terms, policies) must not leak from a previous schedule
  RBT_CUDA(h, cudaMemset(h->buf[RBT_BUF_RIC], 0, size_t(h->buf.doubles(RBT_BUF_RIC, n_grid)) * 8));
  RBT_CUDA(h, cudaMemset(h->buf[RBT_BUF_DIR], 0, size_t(h->buf.doubles(RBT_BUF_DIR, n_grid)) * 8));
  h->n_grid = n_grid;
  h->max_dts0 = max_dts0;
  h->ctrl.assign(ctrl, ctrl + n_grid);
  h->wire_dirty = true;
  return RBT_OK;
}

long long rbt_buf_doubles(rbt_handle* h, int which) {
  if (!h || (which >= RBT_BUF_LIN && !h->stage_ready)) return -1;
  return h->buf.doubles(which, h->n_grid);
}

double* rbt_dev_ptr(rbt_handle* h, int which) { return h ? h->buf[which] : nullptr; }

int rbt_bind_buffer(rbt_handle* h, int which, double* dev) {
  if (!h) return RBT_ERR_ARG;
  // STEPS, PERF and INFO stay the handle's own
  if (which < 0 || which > RBT_BUF_XDIR || which == RBT_BUF_INFO || (which >= RBT_BUF_LIN && !h->stage_ready)) return RBT_ERR_ARG;
  double* q = dev ? dev : h->buf.e[which].own.get();
  if ((reinterpret_cast<uintptr_t>(q) & 15u) != 0) {
    h->err = "[rbt_bind_buffer] invalid argument: device buffer must be 16-byte aligned";
    return RBT_ERR_ARG;
  }
  h->buf.e[which].ptr = q;
  return RBT_OK;
}

// the STO section of the linearization records is read on switching-time stages only (riccati_backward.cuh: cs.sto)
static int ctrl_has_sto(const rbt_stage_ctrl* ctrl, int n_grid) {
  for (int i = 0; i < n_grid; ++i)
    if (ctrl[i].sto || ctrl[i].sto_next) return 1;
  return 0;
}
// wire layouts of all grid points of a schedule; returns the OCP stride in doubles
static long long make_wire_layouts(const rbt_stage_layout& S, const rbt_stage_ctrl* ctrl, int n_grid, int cost_structure,
                                   std::vector<rbt_wire_layout>& out) {
  const int with_sto = ctrl_has_sto(ctrl, n_grid);
  out.resize(n_grid);
  long long off = 0;
  for (int i = 0; i < n_grid; ++i) {
    rbt_make_wire_layout(&S, &ctrl[i], with_sto, cost_structure, &out[i]);
    out[i].ocp_off = int(off);
    off += out[i].w_doubles;
  }
  return off;
}
static int ensure_wire_layouts(rbt_handle* h) {  // rebuilt only when the schedule or the cost structure changed
  if (!h->wire_dirty && h->d_W) return RBT_OK;
  h->w_ocp = make_wire_layouts(h->S, h->ctrl.data(), h->n_grid, h->cost_structure, h->Wv);
  if (!h->d_W) RBT_CUDA(h, dev_alloc(h->d_W, h->n_grid_max));
  RBT_CUDA(h, cudaMemcpy(h->d_W.get(), h->Wv.data(), size_t(h->n_grid) * sizeof(rbt_wire_layout), cudaMemcpyHostToDevice));
  h->wire_dirty = false;
  return RBT_OK;
}

// ---- host <-> device transfers -----------------------------------------------------------------------------------
// The host arrays a transfer plan reads or writes.  Each has the layout of the device buffer it is copied to or from.
enum HostArg { A_KKT, A_LIN, A_WIRE, A_RES, A_CON, A_SOL, A_DX0, A_SOL_OUT, A_CON_OUT, A_STEPS_OUT, N_HOST_ARGS };
// What crosses PCIe in rbt_iteration_host (DENSE), rbt_iteration_host_wire (WIRE) and rbt_iteration_host_resident (RESIDENT).
enum HostMode { DENSE = 0, WIRE = 1, RESIDENT = 2 };

namespace {
// One copy: `rows` rows of `width` doubles, `pitch` doubles apart, starting `off` doubles into the device buffer `dev` and
// into the host array `arg`.
struct Copy {
  cudaMemcpyKind kind;
  int arg;
  double* dev;
  size_t off, pitch, width, rows;
};

// Builds the copies of the batch window `w`.  Only what the kernels read or what persists crosses PCIe: record padding
// never does, the switching-constraint and STO sections only for the stages that carry them.
struct Plan {
  const rbt_handle* h;
  Win w;
  std::vector<Copy> c;

  // the section [off, off + width) of the records (`stride` doubles each) of every grid point of the window
  void records(cudaMemcpyKind k, int arg, double* dev, size_t stride, size_t off, size_t width) {
    const size_t g = size_t(h->n_grid);
    c.push_back({k, arg, dev, size_t(w.b0) * g * stride + off, stride, width, size_t(w.nb) * g});
  }
  // n doubles per OCP of the window
  void per_ocp(cudaMemcpyKind k, int arg, double* dev, size_t n) {
    c.push_back({k, arg, dev, size_t(w.b0) * n, n, n, size_t(w.nb)});
  }
  // the section [off, off + width) of the records of grid point i of every OCP of the window
  void grid_point(int arg, double* dev, size_t stride, int i, size_t off, size_t width) {
    const size_t pitch = size_t(h->n_grid) * stride;
    c.push_back({cudaMemcpyHostToDevice, arg, dev, size_t(w.b0) * pitch + size_t(i) * stride + off, pitch, width, size_t(w.nb)});
  }
  // KKT records: the core section [Fxx|Fvu|Fx|lx|lu|Qxx|Qxu|Quu] of every record, plus the extras of the stages that carry
  // them (switching constraint, STO)
  void kkt() {
    const rbt_layout& L = h->L;
    int n_extra = 0;
    for (const auto& q : h->ctrl) n_extra += (q.ns > 0 || q.sto) ? 1 : 0;
    const bool wide = n_extra * 2 > h->n_grid;  // most stages carry extras (STO horizons): copy core+extras in one go
    records(cudaMemcpyHostToDevice, A_KKT, h->buf[RBT_BUF_KKT], L.k_stride, 0, wide ? L.k_core_size + L.k_extra_size : L.k_core_size);
    if (wide) return;
    for (int i = 0; i < h->n_grid; ++i)
      if (h->ctrl[i].ns > 0 || h->ctrl[i].sto) grid_point(A_KKT, h->buf[RBT_BUF_KKT], L.k_stride, i, L.k_Phix, L.k_extra_size);
  }
  // the switching-constraint sections (Phix, Phia, p, Phit) of the linearization records
  void switching() {
    const rbt_stage_layout& S = h->S;
    for (int i = 0; i < h->n_grid; ++i)
      if (h->ctrl[i].ns > 0 && h->ctrl[i].type != RBT_IMPACT)
        grid_point(A_LIN, h->buf[RBT_BUF_LIN], S.l_stride, i, S.l_Phix, S.l_ha - S.l_Phix);
  }
  void lin() {
    const rbt_stage_layout& S = h->S;
    records(cudaMemcpyHostToDevice, A_LIN, h->buf[RBT_BUF_LIN], S.l_stride, 0, S.l_Phix);  // M .. se3
    records(cudaMemcpyHostToDevice, A_LIN, h->buf[RBT_BUF_LIN], S.l_stride, S.l_ha,        // ha .. dgdf
            size_t(S.l_dgdf) + ((15 * S.ncon + 1) & ~1) - S.l_ha);
    switching();
  }
  // PDIPM records: slack | dual | residual go up, slack | dual come back
  void con(cudaMemcpyKind k, int arg) {
    const rbt_stage_layout& S = h->S;
    records(k, arg, h->buf[RBT_BUF_CON], S.c_stride, S.c_slack, size_t(k == cudaMemcpyHostToDevice ? 3 : 2) * S.ncp);
  }
  // whole records incl. the few padding doubles: ONE contiguous DMA instead of a strided 2-D copy of 1.4 KB rows (the copy
  // engine spends as long per row as on ~4 KB of payload)
  void sol(cudaMemcpyKind k, int arg) { records(k, arg, h->buf[RBT_BUF_SOL], h->S.s_stride, 0, h->S.s_stride); }
  void dx0() { per_ocp(cudaMemcpyHostToDevice, A_DX0, h->buf[RBT_BUF_DX0], h->L.nx); }
};

// rbt_upload(which) of the whole batch
std::vector<Copy> upload_plan(const rbt_handle* h, int which) {
  Plan p{h, {0, h->batch}, {}};
  if (which == RBT_BUF_KKT) p.kkt();
  if (which == RBT_BUF_LIN) p.lin();
  if (which == RBT_BUF_CON) p.con(cudaMemcpyHostToDevice, A_CON);
  if (which == RBT_BUF_SOL) p.sol(cudaMemcpyHostToDevice, A_SOL);
  if (which == RBT_BUF_DX0) p.dx0();
  return p.c;
}

// one rbt_iteration_host* call on the batch window w (the wire modes need ensure_wire_layouts first)
std::vector<Copy> host_plan(const rbt_handle* h, HostMode mode, Win w) {
  const rbt_stage_layout& S = h->S;
  Plan p{h, w, {}};
  if (mode == DENSE) {
    p.lin();
  } else {
    p.per_ocp(cudaMemcpyHostToDevice, A_WIRE, h->d_wire.get(), h->w_ocp);  // packed wire records
    p.switching();
  }
  if (mode == RESIDENT) {  // compact PDIPM residuals [batch][n_grid][ncp] (unpack_wire_kernel scatters them into c_res)
    p.records(cudaMemcpyHostToDevice, A_RES, h->d_res_stage.get(), S.ncp, 0, S.ncp);
  } else {
    p.con(cudaMemcpyHostToDevice, A_CON);
    p.sol(cudaMemcpyHostToDevice, A_SOL);
  }
  p.dx0();
  p.sol(cudaMemcpyDeviceToHost, A_SOL_OUT);
  if (mode == RESIDENT)  // compact slack | dual [batch][n_grid][2 ncp] (packed by pack_slack_dual_kernel)
    p.records(cudaMemcpyDeviceToHost, A_CON_OUT, h->d_sd_stage.get(), 2 * S.ncp, 0, 2 * S.ncp);
  else
    p.con(cudaMemcpyDeviceToHost, A_CON_OUT);
  p.per_ocp(cudaMemcpyDeviceToHost, A_STEPS_OUT, h->buf[RBT_BUF_STEPS], 2);
  return p.c;
}

long long plan_bytes(const std::vector<Copy>& plan, cudaMemcpyKind k) {
  long long bytes = 0;
  for (const Copy& c : plan)
    if (c.kind == k) bytes += (long long)(c.width * c.rows * 8);
  return bytes;
}

int issue(rbt_handle* h, const Copy& c, const double* host_in, double* host_out, cudaStream_t st) {
  const bool up = c.kind == cudaMemcpyHostToDevice;
  void* dst = up ? static_cast<void*>(c.dev + c.off) : static_cast<void*>(host_out + c.off);
  const void* src = up ? static_cast<const void*>(host_in + c.off) : static_cast<const void*>(c.dev + c.off);
  if (c.pitch == c.width)  // contiguous: one linear DMA
    RBT_CUDA(h, cudaMemcpyAsync(dst, src, c.width * c.rows * 8, c.kind, st));
  else
    RBT_CUDA(h, cudaMemcpy2DAsync(dst, c.pitch * 8, src, c.pitch * 8, c.width * 8, c.rows, c.kind, st));
  return RBT_OK;
}
}  // namespace

long long rbt_upload_bytes(rbt_handle* h, int which) {
  if (!h || h->n_grid == 0) return -1;
  const bool stage_buf = which == RBT_BUF_LIN || which == RBT_BUF_CON || which == RBT_BUF_SOL;
  if (!(which == RBT_BUF_KKT || which == RBT_BUF_DX0 || (stage_buf && h->stage_ready))) return -1;
  return plan_bytes(upload_plan(h, which), cudaMemcpyHostToDevice);
}

int rbt_upload(rbt_handle* h, int which, const double* host, void* stream) {
  if (!h || !host) return RBT_ERR_ARG;
  if (which != RBT_BUF_KKT && which != RBT_BUF_DX0 && which != RBT_BUF_LIN && which != RBT_BUF_CON && which != RBT_BUF_SOL)
    return RBT_ERR_ARG;
  if (which >= RBT_BUF_LIN && !h->stage_ready) return RBT_ERR_STATE;
  if (h->n_grid == 0) return RBT_ERR_STATE;
  RBT_CUDA(h, cudaSetDevice(h->device));
  if (which == RBT_BUF_KKT) h->kkt_from_condense = false;
  for (const Copy& c : upload_plan(h, which))
    if (int rc = issue(h, c, host, nullptr, (cudaStream_t)stream)) return rc;
  return RBT_OK;
}

int rbt_download(rbt_handle* h, int which, double* host, void* stream) {
  if (!h || !host || !h->buf[which]) return RBT_ERR_ARG;
  if (h->n_grid == 0) return RBT_ERR_STATE;
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaMemcpyAsync(host, h->buf[which], size_t(rbt_buf_doubles(h, which)) * 8, cudaMemcpyDeviceToHost,
                              (cudaStream_t)stream));
  return RBT_OK;
}

int rbt_download_info(rbt_handle* h, int* host_flags, void* stream) {
  if (!h || !host_flags) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaMemcpyAsync(host_flags, h->d_info.get(), size_t(h->batch) * sizeof(int), cudaMemcpyDeviceToHost,
                              (cudaStream_t)stream));
  return RBT_OK;
}

int rbt_check_info(rbt_handle* h, int* first_bad, void* stream) {
  if (!h) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  std::vector<int> flags(size_t(h->batch), 0);
  RBT_CUDA(h, cudaMemcpyAsync(flags.data(), h->d_info.get(), flags.size() * sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  RBT_CUDA(h, cudaStreamSynchronize((cudaStream_t)stream));
  if (first_bad) *first_bad = -1;
  for (int b = 0; b < h->batch; ++b)
    if (flags[size_t(b)]) {
      if (first_bad) *first_bad = b;
      h->err = "numerical failure: OCP " + std::to_string(b) + " flag " + std::to_string(flags[size_t(b)]) +
               " (1: Quu + B^T P B not positive definite, 2: switching-constraint Schur complement, 4: M, 8: J M^-1 J^T in the condensing)";
      return RBT_ERR_NUMERIC;
    }
  return RBT_OK;
}

static int launch_backward(rbt_handle* h, Win w, int write_fact, cudaStream_t st) {
  constexpr int NP = 6;
  using C = rbt::BwdCfg<INST_NV, INST_NU, INST_NS, NP>;
  if (C::STAGE != h->L.k_stage_size || C::EXTRA != h->L.k_extra_size) {
    h->err = "internal: shared-memory staging size does not match rbt_layout";
    return RBT_ERR_STATE;
  }
  auto kern_s = rbt::riccati_backward_kernel<INST_NV, INST_NU, INST_NS, NP, true>;   // Fqq = I, Fqv = dt I outside the floating-base blocks
  auto kern_g = rbt::riccati_backward_kernel<INST_NV, INST_NU, INST_NS, NP, false>;  // any Fxx
  if (!h->attr_bwd) {  // the attribute is per device: tracked per handle (a handle lives on one device)
    RBT_CUDA(h, cudaFuncSetAttribute(kern_s, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES));
    RBT_CUDA(h, cudaFuncSetAttribute(kern_g, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES));
    h->attr_bwd = true;
  }
  rbt::BwdParams p;
  p.L = h->L;
  p.ctrl = h->d_ctrl.get();
  const size_t go = size_t(w.b0) * h->n_grid;
  p.n_grid = h->n_grid;
  p.batch = w.nb;
  p.max_dts0 = h->max_dts0;
  p.kkt = h->buf[RBT_BUF_KKT] + go * h->L.k_stride;
  p.ric = h->buf[RBT_BUF_RIC] + go * h->L.r_stride;
  p.fact = write_fact ? h->buf[RBT_BUF_FACT] + go * h->L.f_stride : nullptr;
  p.info = h->d_info.get() + w.b0;
  p.struct_flag = nullptr;
  if (!h->keep_info) RBT_CUDA(h, cudaMemsetAsync(p.info, 0, size_t(w.nb) * sizeof(int), st));
  h->keep_info = false;
  // Which instance: the condensing kernel writes Fqq = I, Fqv = dt I outside the floating-base blocks by construction
  // (state_equation.cpp:52-55,68-87), a caller can declare it (rbt_set_fxx_structure), otherwise (RBT_FXX_AUTO) the records are
  // inspected on the device and BOTH instances are launched -- the one the flag does not select returns at once.
  const bool known_struct = h->kkt_from_condense || h->fxx_mode == RBT_FXX_MECHANICAL;
  h->kkt_from_condense = false;
  if (known_struct) {
    kern_s<<<w.nb, C::NTHREADS, C::SMEM_BYTES, st>>>(p);
    h->launches += 1;
  } else if (h->fxx_mode == RBT_FXX_GENERAL) {
    kern_g<<<w.nb, C::NTHREADS, C::SMEM_BYTES, st>>>(p);
    h->launches += 1;
  } else {
    RBT_CUDA(h, cudaMemsetAsync(h->d_struct.get(), 0, 2 * sizeof(int), st));
    rbt::check_fxx_structure_kernel<INST_NV, NP><<<(w.nb * (h->n_grid - 1) + 7) / 8, 256, 0, st>>>(p, h->d_struct.get());
    p.struct_flag = h->d_struct.get();
    kern_s<<<w.nb, C::NTHREADS, C::SMEM_BYTES, st>>>(p);
    kern_g<<<w.nb, C::NTHREADS, C::SMEM_BYTES, st>>>(p);
    h->launches += 3;
  }
  RBT_CUDA(h, cudaGetLastError());
  return RBT_OK;
}

int rbt_set_fxx_structure(rbt_handle* h, int mode) {
  if (!h || (mode != RBT_FXX_AUTO && mode != RBT_FXX_MECHANICAL && mode != RBT_FXX_GENERAL)) return RBT_ERR_ARG;
  h->fxx_mode = mode;
  return RBT_OK;
}

static int launch_forward(rbt_handle* h, Win w, cudaStream_t st) {
  using C = rbt::FwdCfg<INST_NV, INST_NU, INST_NS>;
  auto kern = rbt::riccati_forward_kernel<INST_NV, INST_NU, INST_NS>;
  if (!h->attr_fwd) {
    RBT_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES));
    h->attr_fwd = true;
  }
  rbt::FwdParams p;
  p.L = h->L;
  p.ctrl = h->d_ctrl.get();
  const size_t go = size_t(w.b0) * h->n_grid;
  p.n_grid = h->n_grid;
  p.batch = w.nb;
  p.kkt = h->buf[RBT_BUF_KKT] + go * h->L.k_stride;
  p.ric = h->buf[RBT_BUF_RIC] + go * h->L.r_stride;
  p.dx0 = h->buf[RBT_BUF_DX0] + size_t(w.b0) * h->L.nx;
  p.dir = h->buf[RBT_BUF_DIR] + go * h->L.d_stride;
  kern<<<w.nb, C::NTHREADS, C::SMEM_BYTES, st>>>(p);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_riccati_backward(rbt_handle* h, int write_fact, void* stream) {
  if (!h) return RBT_ERR_ARG;
  if (h->n_grid == 0) {
    h->err = "[rbt_riccati_backward] no schedule set";
    return RBT_ERR_STATE;
  }
  RBT_CUDA(h, cudaSetDevice(h->device));
  return launch_backward(h, {0, h->batch}, write_fact, (cudaStream_t)stream);
}

int rbt_riccati_forward(rbt_handle* h, void* stream) {
  if (!h) return RBT_ERR_ARG;
  if (h->n_grid == 0) {
    h->err = "[rbt_riccati_forward] no schedule set";
    return RBT_ERR_STATE;
  }
  RBT_CUDA(h, cudaSetDevice(h->device));
  return launch_forward(h, {0, h->batch}, (cudaStream_t)stream);
}

// ---- stage layer ---------------------------------------------------------------------------------------------------
int rbt_stage_layout_get(const rbt_stage_dims* sdims, const char* field) {
  if (!sdims || !field) return -1;
  rbt_stage_layout S;
  rbt_make_stage_layout(sdims, &S);
  return rbt_stage_layout_field(&S, field);
}

int rbt_stage_setup(rbt_handle* h, const rbt_stage_dims* sd, const rbt_constraint_table* table) {
  if (!h || !sd || !table) return RBT_ERR_ARG;
  if (sd->nv != h->dims.nv || sd->nu != h->dims.nu || sd->ns_max != h->dims.ns_max || sd->n_passive != h->dims.n_passive ||
      sd->n_passive != sd->nv - sd->nu /* dim_passive = dimv - dimu (robot.cpp): compiled into the stage kernels */ ||
      sd->nf_max != 12 || table->n_box != sd->n_box || table->n_contacts != sd->n_contacts || sd->n_box > RBT_MAX_BOX_ROWS ||
      sd->n_contacts > RBT_MAX_CONTACTS || !(table->barrier > 0) || !(table->fraction_to_boundary > 0) ||
      !(table->fraction_to_boundary <= 1)) {
    h->err = "[rbt_stage_setup] invalid argument: stage dims / constraint table inconsistent with the handle";
    return RBT_ERR_ARG;
  }
  for (int r = 0; r < table->n_box; ++r) {
    const rbt_box_row& b = table->box[r];
    const int lim = (b.var == RBT_VAR_U) ? sd->nu : sd->nv;
    if (b.var < 0 || b.var > 3 || b.idx < 0 || b.idx >= lim || (b.sign != 1 && b.sign != -1)) {
      h->err = "[rbt_stage_setup] invalid argument: bad box row " + std::to_string(r);
      return RBT_ERR_ARG;
    }
  }
  {
    if (3 * sd->nv + sd->nu > RBT_MAX_TARGETS) {
      h->err = "[rbt_stage_setup] invalid argument: too many limit targets";
      return RBT_ERR_ARG;
    }
    std::vector<int> cnt(RBT_MAX_TARGETS, 0);
    for (int r = 0; r < table->n_box; ++r) {
      const rbt_box_row& b = table->box[r];
      const int t = (b.var == RBT_VAR_U) ? 3 * sd->nv + b.idx : b.var * sd->nv + b.idx;
      if (++cnt[t] > 4) {
        h->err = "[rbt_stage_setup] invalid argument: more than 4 box rows on one variable";
        return RBT_ERR_ARG;
      }
    }
  }
  if (h->stage_ready) {  // a second call would replace stage buffers the caller may have re-bound
    h->err = "[rbt_stage_setup] already set up on this handle (create a new handle for another constraint table)";
    return RBT_ERR_STATE;
  }
  h->sdims = *sd;
  h->table = *table;
  h->stage_ready = true;  // (for check_contacts; reset below on failure)
  if (h->n_grid > 0 && check_contacts(h, h->ctrl.data(), h->n_grid) != RBT_OK) {
    h->stage_ready = false;
    return RBT_ERR_ARG;
  }
  h->stage_ready = false;
  rbt_make_stage_layout(sd, &h->S);
  {  // condense_kernel lands [l_D, l_Phix) and [l_ha, l_dgdq) of the record in place: the static mirror must match
    using C = rbt::CondCfg<INST_NV, INST_NU, INST_NS>;
    const rbt_stage_layout& S = h->S;
    const int gsz = (S.l_dgdf - S.l_dgdq) + ((15 * S.ncon + 1) & ~1);
    const int q0 = S.l_Quu - C::IN1A;  // record offset that maps onto the second in-place mirror
    const bool ok = S.l_Qxx - S.l_D == C::IN1A && S.l_Phix - S.l_Quu == C::IN1B && S.l_IDC - S.l_D == C::i_IDC &&
                    S.l_Qaa - S.l_D == C::i_Qaa && S.l_Qff - S.l_D == C::i_Qff && S.l_Qqf - S.l_D == C::i_Qqf &&
                    S.l_lx - q0 == C::i_lx && S.l_la - q0 == C::i_la && S.l_lf - q0 == C::i_lf && S.l_lu - q0 == C::i_lu &&
                    S.l_Fx - q0 == C::i_Fx && S.l_lup - q0 == C::i_lup && S.l_se3 - q0 == C::i_se3 && S.l_dgdq - S.l_ha == C::IN2 &&
                    S.l_hf - S.l_ha == C::j_hf && S.l_hx - S.l_ha == C::j_hx && S.l_hu - S.l_ha == C::j_hu &&
                    S.l_fx - S.l_ha == C::j_fx && S.l_sc - S.l_ha == C::j_sc &&
                    5 * S.ncp + gsz <= C::NVF * C::NX &&  // PDIPM staging fits in the R buffer
                    S.l_J - S.l_M == rbt::MjtjCfg<INST_NV, INST_NU>::o_J && S.l_D - S.l_M == rbt::MjtjCfg<INST_NV, INST_NU>::MJ;
    if (!ok) {
      h->err = "[rbt_stage_setup] invalid argument: stage layout not supported by the compiled condensing kernel";
      return RBT_ERR_ARG;
    }
  }
  if (h->S.ncp > 160 || h->S.l_stride - h->S.l_dgdq > 512) {  // shared-memory staging areas of expand_kernel
    h->err = "[rbt_stage_setup] invalid argument: more than 160 inequality rows or more than 4 friction cones";
    return RBT_ERR_ARG;
  }
  RBT_CUDA(h, cudaSetDevice(h->device));
  // uploads skip record padding: the zeroed allocation keeps it defined
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_LIN, h->S.l_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_CON, h->S.c_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_EXP, h->S.e_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_SOL, h->S.s_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_XDIR, h->S.x_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_STEPS, 2, false));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_PERF, 8, false));
  RBT_CUDA(h, dev_alloc(h->d_ones, size_t(h->batch) * 2));
  RBT_CUDA(h, dev_alloc(h->d_stage_perf, size_t(h->batch) * h->n_grid_max * 4));
  RBT_CUDA(h, dev_alloc(h->d_x0in, size_t(h->batch) * 2 * h->dims.nv));
  {  // box rows acting on each target entry (var, idx), in ascending row order (deterministic accumulation on the device):
     // entry = (row + 1) * sign, 0 = none.  Device memory, not kernel parameters: the lanes of a warp look up different targets,
     // and a divergent constant-bank access is serialised.
    int tg[RBT_MAX_TARGETS][4] = {};
    for (int r = 0; r < h->table.n_box; ++r) {
      const rbt_box_row& b = h->table.box[r];
      const int t = (b.var == RBT_VAR_U) ? 3 * h->sdims.nv + b.idx : b.var * h->sdims.nv + b.idx;
      for (int q = 0; q < 4; ++q)
        if (tg[t][q] == 0) {
          tg[t][q] = (r + 1) * (b.sign < 0 ? -1 : 1);
          break;
        }
    }
    // ... followed by the level of every box row (2 = position, 1 = velocity, 0 = acceleration / torque): a row acts on a grid
    // point iff level + ineq_gate <= 2 (ConstraintsData::setTimeStage)
    int lvl[RBT_MAX_BOX_ROWS] = {};
    for (int r = 0; r < h->table.n_box; ++r) lvl[r] = h->table.box[r].var == RBT_VAR_Q ? 2 : (h->table.box[r].var == RBT_VAR_V ? 1 : 0);
    RBT_CUDA(h, dev_alloc(h->d_tgt, sizeof(tg) / sizeof(int) + sizeof(lvl) / sizeof(int)));
    RBT_CUDA(h, cudaMemcpy(h->d_tgt.get(), tg, sizeof(tg), cudaMemcpyHostToDevice));
    RBT_CUDA(h, cudaMemcpy(h->d_tgt.get() + RBT_MAX_TARGETS * 4, lvl, sizeof(lvl), cudaMemcpyHostToDevice));
  }
  std::vector<double> ones(size_t(h->batch) * 2, 1.0);
  RBT_CUDA(h, cudaMemcpy(h->d_ones.get(), ones.data(), ones.size() * 8, cudaMemcpyHostToDevice));
  RBT_CUDA(h, cudaMemcpy(h->buf[RBT_BUF_STEPS], ones.data(), ones.size() * 8, cudaMemcpyHostToDevice));
  h->stage_ready = true;
  return RBT_OK;
}

static rbt::StageParams make_stage_params(rbt_handle* h, Win w) {
  rbt::StageParams p;
  p.K = h->L;
  p.S = h->S;
  p.tab = h->table;
  p.ctrl = h->d_ctrl.get();
  const size_t go = size_t(w.b0) * h->n_grid;
  p.n_grid = h->n_grid;
  p.batch = w.nb;
  p.lin = h->buf[RBT_BUF_LIN] + go * h->S.l_stride;
  p.con = h->buf[RBT_BUF_CON] + go * h->S.c_stride;
  p.kkt = h->buf[RBT_BUF_KKT] + go * h->L.k_stride;
  p.ex = h->buf[RBT_BUF_EXP] + go * h->S.e_stride;
  p.dir = h->buf[RBT_BUF_DIR] + go * h->L.d_stride;
  p.xd = h->buf[RBT_BUF_XDIR] + go * h->S.x_stride;
  p.sol = h->buf[RBT_BUF_SOL] + go * h->S.s_stride;
  p.steps = h->buf[RBT_BUF_STEPS] + 2 * size_t(w.b0);
  p.info = h->d_info.get() + w.b0;
  p.tgt = reinterpret_cast<const int4*>(h->d_tgt.get());
  p.row_level = h->d_tgt.get() + RBT_MAX_TARGETS * 4;
  return p;
}

static int launch_condense(rbt_handle* h, Win w, cudaStream_t st) {
  using C = rbt::CondCfg<INST_NV, INST_NU, INST_NS>;
  auto kern = rbt::condense_kernel<INST_NV, INST_NU, INST_NS>;
  if (!h->attr_cond) {
    RBT_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES));
    h->attr_cond = true;
  }
  const rbt::StageParams p = make_stage_params(h, w);
  RBT_CUDA(h, cudaMemsetAsync(p.info, 0, size_t(w.nb) * sizeof(int), st));
  rbt::mjtjinv_kernel<INST_NV, INST_NU><<<(w.nb * h->n_grid + 1) / 2, 64, 0, st>>>(p);  // K1: Z = [[M,J^T],[J,0]]^-1
  RBT_CUDA(h, cudaGetLastError());
  if (h->ev_condense_mid) RBT_CUDA(h, cudaEventRecord(h->ev_condense_mid, st));
  kern<<<w.nb * h->n_grid, C::NTHREADS, C::SMEM_BYTES, st>>>(p);                      // K2: condensing (DMMA)
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 2;
  h->keep_info = true;
  h->kkt_from_condense = true;
  return RBT_OK;
}

static int launch_expand(rbt_handle* h, Win w, cudaStream_t st) {
  const rbt::StageParams p = make_stage_params(h, w);
  RBT_CUDA(h, cudaMemcpyAsync(p.steps, h->d_ones.get(), size_t(w.nb) * 2 * 8, cudaMemcpyDeviceToDevice, st));
  rbt::expand_kernel<INST_NV, INST_NU, INST_NS><<<w.nb * h->n_grid, rbt::XTHR, 0, st>>>(p);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

static int launch_update(rbt_handle* h, Win w, cudaStream_t st) {
  rbt::update_kernel<INST_NV, INST_NU, INST_NS><<<w.nb * h->n_grid, rbt::XTHR, 0, st>>>(make_stage_params(h, w));
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

#define RBT_STAGE_CHECK(h, what)                                  \
  if (!(h)) return RBT_ERR_ARG;                                   \
  if (!(h)->stage_ready || (h)->n_grid == 0) {                    \
    (h)->err = "[" what "] stage layer not set up / no schedule"; \
    return RBT_ERR_STATE;                                         \
  }                                                               \
  RBT_CUDA(h, cudaSetDevice((h)->device));

int rbt_condense(rbt_handle* h, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_condense");
  return launch_condense(h, {0, h->batch}, (cudaStream_t)stream);
}

int rbt_set_condense_event(rbt_handle* h, void* cuda_event) {
  if (!h) return RBT_ERR_ARG;
  h->ev_condense_mid = (cudaEvent_t)cuda_event;
  return RBT_OK;
}

int rbt_expand_and_step_sizes(rbt_handle* h, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_expand_and_step_sizes");
  return launch_expand(h, {0, h->batch}, (cudaStream_t)stream);
}

int rbt_update(rbt_handle* h, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_update");
  return launch_update(h, {0, h->batch}, (cudaStream_t)stream);
}

// the whole batch
static rbt::EvalParams make_eval_params(rbt_handle* h) {
  rbt::EvalParams q;
  q.sp = make_stage_params(h, {0, h->batch});
  q.stage_perf = h->d_stage_perf.get();
  q.perf = h->buf[RBT_BUF_PERF];
  q.x0in = h->d_x0in.get();
  q.dx0 = h->buf[RBT_BUF_DX0];
  return q;
}

int rbt_eval_kkt(rbt_handle* h, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_eval_kkt");
  cudaStream_t st = (cudaStream_t)stream;
  const rbt::EvalParams q = make_eval_params(h);
  rbt::perf_index_kernel<<<(h->batch * h->n_grid + 3) / 4, 128, 0, st>>>(q);
  rbt::perf_reduce_kernel<<<(h->batch + 127) / 128, 128, 0, st>>>(q);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 2;
  return RBT_OK;
}

int rbt_set_slack_and_dual_positive(rbt_handle* h, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_set_slack_and_dual_positive");
  const rbt::EvalParams q = make_eval_params(h);
  const long long total = (long long)h->batch * h->n_grid * h->S.ncp;
  rbt::slack_dual_positive_kernel<<<unsigned((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(q);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_set_joint_limits(rbt_handle* h, const double* bound_host) {
  if (!h || !bound_host) return RBT_ERR_ARG;
  if (!h->stage_ready) {
    h->err = "[rbt_set_joint_limits] stage layer not set up";
    return RBT_ERR_STATE;
  }
  RBT_CUDA(h, cudaSetDevice(h->device));
  if (!h->d_bound) RBT_CUDA(h, dev_alloc(h->d_bound, RBT_MAX_BOX_ROWS));
  RBT_CUDA(h, cudaMemcpy(h->d_bound.get(), bound_host, sizeof(double) * h->table.n_box, cudaMemcpyHostToDevice));
  return RBT_OK;
}

int rbt_linearize_joint_limits(rbt_handle* h, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_linearize_joint_limits");
  if (!h->d_bound) {
    h->err = "[rbt_linearize_joint_limits] call rbt_set_joint_limits first";
    return RBT_ERR_STATE;
  }
  const rbt::EvalParams q = make_eval_params(h);
  const long long total = (long long)h->batch * h->n_grid * (3 * h->S.nv + h->S.nu);
  rbt::linearize_joint_limits_kernel<<<unsigned((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(q, h->d_bound.get());
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_initial_state_direction(rbt_handle* h, const double* dq0_v0_host, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_initial_state_direction");
  if (!dq0_v0_host) return RBT_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  RBT_CUDA(h, cudaMemcpyAsync(h->d_x0in.get(), dq0_v0_host, size_t(h->batch) * 2 * h->dims.nv * 8, cudaMemcpyHostToDevice, st));
  const rbt::EvalParams q = make_eval_params(h);
  const int total = h->batch * h->L.nx;
  rbt::initial_state_direction_kernel<<<(total + 127) / 128, 128, 0, st>>>(q);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

// ---- line search: trial step sizes as an extra batch axis -------------------------------------------------------------------
enum { RBT_LS_FILTER_CAP = 16 };

static int ls_ensure(rbt_handle* h, int n_trials) {
  if (n_trials <= h->ls_trials) return RBT_OK;
  const size_t kb = size_t(n_trials) * h->batch;
  RBT_CUDA(h, dev_alloc(h->d_ls_alphas, kb));
  RBT_CUDA(h, dev_alloc(h->d_ls_barrier, kb));
  RBT_CUDA(h, dev_alloc(h->d_ls_stage_barrier, kb * h->n_grid_max));
  RBT_CUDA(h, dev_alloc(h->d_ls_trial, kb * h->n_grid_max * rbt::T_STRIDE));
  RBT_CUDA(h, dev_alloc(h->d_ls_in, 2 * kb + 2 * size_t(h->batch)));  // cost | viol of the trials, cost0 | viol0
  if (!h->d_ls_filt) {
    RBT_CUDA(h, dev_alloc(h->d_ls_filt, size_t(h->batch) * 2 * RBT_LS_FILTER_CAP));
    RBT_CUDA(h, dev_alloc(h->d_ls_nfilt, h->batch));
    RBT_CUDA(h, dev_alloc(h->d_ls_step, h->batch));
    RBT_CUDA(h, dev_alloc(h->d_ls_k, h->batch));
    RBT_CUDA(h, cudaMemset(h->d_ls_nfilt.get(), 0, size_t(h->batch) * sizeof(int)));
  }
  h->ls_trials = n_trials;
  return RBT_OK;
}

int rbt_trial_doubles(void) { return rbt::T_STRIDE; }

int rbt_line_search_trials(rbt_handle* h, int n_trials, double step_size_reduction_rate, double* alphas_host, double* barrier_host,
                           double* trial_host, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_line_search_trials");
  if (n_trials < 1 || n_trials > 64 || !(step_size_reduction_rate > 0.0 && step_size_reduction_rate < 1.0)) {
    h->err = "[rbt_line_search_trials] invalid argument: 1 <= n_trials <= 64, 0 < step_size_reduction_rate < 1";
    return RBT_ERR_ARG;
  }
  if (int rc = ls_ensure(h, n_trials)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  rbt::TrialParams q;
  q.sp = make_stage_params(h, {0, h->batch});
  q.n_trials = n_trials;
  q.rate = step_size_reduction_rate;
  q.alphas = h->d_ls_alphas.get();
  q.trial = h->d_ls_trial.get();
  q.stage_barrier = h->d_ls_stage_barrier.get();
  q.barrier = h->d_ls_barrier.get();
  const long long warps = (long long)n_trials * h->batch * h->n_grid;
  rbt::trial_solution_kernel<<<unsigned((warps + 3) / 4), 128, 0, st>>>(q);
  rbt::trial_reduce_kernel<<<(n_trials * h->batch + 127) / 128, 128, 0, st>>>(q);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 2;
  const size_t kb = size_t(n_trials) * h->batch;
  if (alphas_host) RBT_CUDA(h, cudaMemcpyAsync(alphas_host, h->d_ls_alphas.get(), kb * 8, cudaMemcpyDeviceToHost, st));
  if (barrier_host) RBT_CUDA(h, cudaMemcpyAsync(barrier_host, h->d_ls_barrier.get(), kb * 8, cudaMemcpyDeviceToHost, st));
  if (trial_host) RBT_CUDA(h, cudaMemcpyAsync(trial_host, h->d_ls_trial.get(), kb * h->n_grid * rbt::T_STRIDE * 8, cudaMemcpyDeviceToHost, st));
  return RBT_OK;
}

double* rbt_line_search_trial_dev(rbt_handle* h) { return h ? h->d_ls_trial.get() : nullptr; }

int rbt_line_search_clear_history(rbt_handle* h, void* stream) {
  if (!h) return RBT_ERR_ARG;
  if (h->d_ls_nfilt) RBT_CUDA(h, cudaMemsetAsync(h->d_ls_nfilt.get(), 0, size_t(h->batch) * sizeof(int), (cudaStream_t)stream));
  return RBT_OK;
}

int rbt_line_search_filter(rbt_handle* h, int n_trials, double step_size_reduction_rate, double min_step_size,
                           double filter_cost_reduction_rate, double filter_constraint_violation_reduction_rate,
                           const double* cost0_host, const double* violation0_host, const double* cost_host,
                           const double* violation_host, double* step_host, int* accepted_trial_host, void* stream) {
  RBT_STAGE_CHECK(h, "rbt_line_search_filter");
  if (n_trials < 1 || n_trials > h->ls_trials || !cost0_host || !violation0_host || !cost_host || !violation_host ||
      !(filter_cost_reduction_rate > 0.0) || !(filter_constraint_violation_reduction_rate > 0.0)) {
    h->err = "[rbt_line_search_filter] invalid argument (call rbt_line_search_trials with at least n_trials first; the reduction "
             "rates must be positive like LineSearchFilter's, line_search_filter.cpp:15-20)";
    return RBT_ERR_ARG;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t kb = size_t(n_trials) * h->batch;
  double* d_cost = h->d_ls_in.get();
  double* d_viol = d_cost + size_t(h->ls_trials) * h->batch;
  double* d_c0 = d_cost + 2 * size_t(h->ls_trials) * h->batch;
  double* d_v0 = d_c0 + h->batch;
  RBT_CUDA(h, cudaMemcpyAsync(d_cost, cost_host, kb * 8, cudaMemcpyHostToDevice, st));
  RBT_CUDA(h, cudaMemcpyAsync(d_viol, violation_host, kb * 8, cudaMemcpyHostToDevice, st));
  RBT_CUDA(h, cudaMemcpyAsync(d_c0, cost0_host, size_t(h->batch) * 8, cudaMemcpyHostToDevice, st));
  RBT_CUDA(h, cudaMemcpyAsync(d_v0, violation0_host, size_t(h->batch) * 8, cudaMemcpyHostToDevice, st));
  rbt::FilterParams q;
  q.batch = h->batch; q.n_trials = n_trials; q.cap = RBT_LS_FILTER_CAP;
  q.rate = step_size_reduction_rate; q.min_step = min_step_size;
  q.cost_rate = filter_cost_reduction_rate; q.viol_rate = filter_constraint_violation_reduction_rate;
  q.steps = h->buf[RBT_BUF_STEPS]; q.cost0 = d_c0; q.viol0 = d_v0; q.cost = d_cost; q.barrier = h->d_ls_barrier.get(); q.viol = d_viol;
  q.filt = h->d_ls_filt.get(); q.nfilt = h->d_ls_nfilt.get(); q.out_step = h->d_ls_step.get(); q.out_k = h->d_ls_k.get();
  rbt::line_search_filter_kernel<<<(h->batch + 127) / 128, 128, 0, st>>>(q);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  if (step_host) RBT_CUDA(h, cudaMemcpyAsync(step_host, h->d_ls_step.get(), size_t(h->batch) * 8, cudaMemcpyDeviceToHost, st));
  if (accepted_trial_host) RBT_CUDA(h, cudaMemcpyAsync(accepted_trial_host, h->d_ls_k.get(), size_t(h->batch) * sizeof(int), cudaMemcpyDeviceToHost, st));
  return RBT_OK;
}

int rbt_iteration_host_bytes(rbt_handle* h, int mode, long long* h2d, long long* d2h) {
  if (!h || !h->stage_ready || h->n_grid == 0) return RBT_ERR_STATE;
  if (mode != DENSE && mode != WIRE && mode != RESIDENT) return RBT_ERR_ARG;
  if (mode != DENSE) {
    RBT_CUDA(h, cudaSetDevice(h->device));
    if (int rc = ensure_wire_layouts(h)) return rc;
  }
  const std::vector<Copy> plan = host_plan(h, HostMode(mode), {0, h->batch});
  if (h2d) *h2d = plan_bytes(plan, cudaMemcpyHostToDevice);
  if (d2h) *d2h = plan_bytes(plan, cudaMemcpyDeviceToHost);
  return RBT_OK;
}

// RESIDENT: solution, slack and dual stay where the previous iteration left them on the device; only the PDIPM residuals
// come from the host, con_host / sol_host are not read.  WIRE, RESIDENT: lin_host holds the switching-constraint sections.
static int iteration_host_impl(rbt_handle* h, HostMode mode, const double* wire_host, const double* lin_host,
                               const double* con_host, const double* sol_host, const double* res_host, const double* dx0_host,
                               double* sol_out, double* con_out, double* steps_out, void* stream) {
  if (!h || (mode == DENSE ? !lin_host : !wire_host) || !dx0_host) return RBT_ERR_ARG;
  if (mode == RESIDENT ? !res_host : (!con_host || !sol_host)) return RBT_ERR_ARG;
  RBT_STAGE_CHECK(h, "rbt_iteration_host");
  if (mode != DENSE) {
    if (int rc = ensure_wire_layouts(h)) return rc;
    bool sw = false;
    for (int i = 0; i < h->n_grid; ++i) sw = sw || (h->ctrl[i].ns > 0 && h->ctrl[i].type != RBT_IMPACT);
    if (sw && !lin_host) {
      h->err = "[rbt_iteration_host_wire] invalid argument: the schedule has switching-constraint stages, their sections come from lin_host_switching";
      return RBT_ERR_ARG;
    }
    if (!h->d_wire) {  // sized for the largest possible record at every grid point
      rbt_wire_layout wmax;
      rbt_stage_ctrl cmax = {};
      cmax.type = RBT_INTERMEDIATE; cmax.nf = h->S.nfm; cmax.contact_mask = (1 << h->S.ncon) - 1;
      rbt_make_wire_layout(&h->S, &cmax, 1, RBT_COST_GENERAL, &wmax);
      RBT_CUDA(h, dev_alloc(h->d_wire, size_t(h->batch) * h->n_grid_max * wmax.w_doubles));
    }
  }
  if (mode == RESIDENT && !h->d_res_stage) {
    RBT_CUDA(h, dev_alloc(h->d_res_stage, size_t(h->batch) * h->n_grid_max * h->S.ncp));
    RBT_CUDA(h, dev_alloc(h->d_sd_stage, size_t(h->batch) * h->n_grid_max * 2 * h->S.ncp));
  }
  const double* in[N_HOST_ARGS] = {};
  double* out[N_HOST_ARGS] = {};
  in[A_WIRE] = wire_host, in[A_LIN] = lin_host, in[A_CON] = con_host, in[A_SOL] = sol_host, in[A_RES] = res_host;
  in[A_DX0] = dx0_host;
  out[A_SOL_OUT] = sol_out, out[A_CON_OUT] = con_out, out[A_STEPS_OUT] = steps_out;
  cudaStream_t st = (cudaStream_t)stream;
  // chunks of the batch: the upload of chunk c+1, the kernels of chunk c and the download of chunk c-1 overlap
  int n_chunks = h->batch >= 512 ? 8 : (h->batch >= 128 ? 4 : 1);
  if (const char* e = getenv("RBT_E2E_CHUNKS")) n_chunks = std::max(1, std::min(atoi(e), h->batch));
  if (!h->s_h2d) {
    cudaStream_t s1, s2;
    RBT_CUDA(h, cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking));
    h->s_h2d.reset(s1);
    RBT_CUDA(h, cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
    h->s_d2h.reset(s2);
  }
  while ((int)h->ev.size() < 2 * n_chunks + 2) {
    cudaEvent_t e;
    RBT_CUDA(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->ev.emplace_back(e);
  }
  cudaStream_t s_h2d = h->s_h2d.get(), s_d2h = h->s_d2h.get();
  cudaEvent_t ev_entry = h->ev[2 * n_chunks].get(), ev_exit = h->ev[2 * n_chunks + 1].get();
  RBT_CUDA(h, cudaEventRecord(ev_entry, st));            // device buffers may still be read by earlier work on `stream`
  RBT_CUDA(h, cudaStreamWaitEvent(s_h2d, ev_entry, 0));
  RBT_CUDA(h, cudaStreamWaitEvent(s_d2h, ev_entry, 0));
  for (int c = 0; c < n_chunks; ++c) {
    const int b0 = int((long long)h->batch * c / n_chunks), b1 = int((long long)h->batch * (c + 1) / n_chunks);
    const Win w{b0, b1 - b0};
    if (w.nb <= 0) continue;
    const std::vector<Copy> plan = host_plan(h, mode, w);
    for (const Copy& k : plan)
      if (k.kind == cudaMemcpyHostToDevice && in[k.arg])
        if (int rc = issue(h, k, in[k.arg], nullptr, s_h2d)) return rc;
    cudaEvent_t ev_up = h->ev[2 * c].get(), ev_done = h->ev[2 * c + 1].get();
    RBT_CUDA(h, cudaEventRecord(ev_up, s_h2d));
    RBT_CUDA(h, cudaStreamWaitEvent(st, ev_up, 0));
    const size_t go = size_t(b0) * h->n_grid;
    if (mode != DENSE) {  // expand the packed records of this chunk into the linearization records
      rbt::WireParams wp;
      wp.W = h->d_W.get();
      wp.n_grid = h->n_grid;
      wp.ocp_stride = h->w_ocp;
      wp.l_stride = h->S.l_stride;
      wp.wire = h->d_wire.get() + size_t(b0) * h->w_ocp;
      wp.lin = h->buf[RBT_BUF_LIN] + go * h->S.l_stride;
      wp.res = mode == RESIDENT ? h->d_res_stage.get() + go * h->S.ncp : nullptr;
      wp.con = h->buf[RBT_BUF_CON] + go * h->S.c_stride;
      wp.c_stride = h->S.c_stride; wp.c_res = h->S.c_res; wp.ncp = h->S.ncp;
      rbt::unpack_wire_kernel<<<w.nb * h->n_grid, 128, 0, st>>>(wp);
      h->launches += 1;
    }
    int rc;
    if ((rc = launch_condense(h, w, st)) || (rc = launch_backward(h, w, 0, st)) || (rc = launch_forward(h, w, st)) ||
        (rc = launch_expand(h, w, st)) || (rc = launch_update(h, w, st)))
      return rc;
    if (mode == RESIDENT && con_out) {
      rbt::pack_slack_dual_kernel<<<w.nb * h->n_grid, 64, 0, st>>>(h->buf[RBT_BUF_CON] + go * h->S.c_stride, h->S.c_stride,
                                                                 h->S.c_slack, 2 * h->S.ncp, h->d_sd_stage.get() + go * 2 * h->S.ncp);
      h->launches += 1;
    }
    RBT_CUDA(h, cudaEventRecord(ev_done, st));
    RBT_CUDA(h, cudaStreamWaitEvent(s_d2h, ev_done, 0));
    for (const Copy& k : plan)
      if (k.kind == cudaMemcpyDeviceToHost && out[k.arg])
        if (int rc2 = issue(h, k, nullptr, out[k.arg], s_d2h)) return rc2;
  }
  RBT_CUDA(h, cudaEventRecord(ev_exit, s_d2h));       // `stream` (what the caller synchronizes) covers the downloads too
  RBT_CUDA(h, cudaStreamWaitEvent(st, ev_exit, 0));
  return RBT_OK;
}

int rbt_iteration_host(rbt_handle* h, const double* lin_host, const double* con_host, const double* sol_host,
                       const double* dx0_host, double* sol_out, double* con_out, double* steps_out, void* stream) {
  return iteration_host_impl(h, DENSE, nullptr, lin_host, con_host, sol_host, nullptr, dx0_host, sol_out, con_out, steps_out,
                             stream);
}

int rbt_iteration_host_wire(rbt_handle* h, const double* wire_host, const double* lin_host_switching, const double* con_host,
                            const double* sol_host, const double* dx0_host, double* sol_out, double* con_out,
                            double* steps_out, void* stream) {
  return iteration_host_impl(h, WIRE, wire_host, lin_host_switching, con_host, sol_host, nullptr, dx0_host, sol_out, con_out,
                             steps_out, stream);
}

int rbt_iteration_host_resident(rbt_handle* h, const double* wire_host, const double* lin_host_switching, const double* res_host,
                                const double* dx0_host, double* sol_out, double* slack_dual_out, double* steps_out, void* stream) {
  return iteration_host_impl(h, RESIDENT, wire_host, lin_host_switching, nullptr, nullptr, res_host, dx0_host, sol_out,
                             slack_dual_out, steps_out, stream);
}

int rbt_set_wire_cost_structure(rbt_handle* h, int cost_structure) {
  if (!h || (cost_structure != RBT_COST_GENERAL && cost_structure != RBT_COST_ROBOTOC)) return RBT_ERR_ARG;
  if (h->cost_structure != cost_structure) h->wire_dirty = true;
  h->cost_structure = cost_structure;
  return RBT_OK;
}

int rbt_wire_doubles(const rbt_stage_dims* sdims, const rbt_stage_ctrl* ctrl, int n_grid, int cost_structure) {
  if (!sdims || !ctrl || n_grid <= 0) return -1;
  rbt_stage_layout S;
  rbt_make_stage_layout(sdims, &S);
  std::vector<rbt_wire_layout> W;
  return int(make_wire_layouts(S, ctrl, n_grid, cost_structure, W));
}

int rbt_wire_layout_get(const rbt_stage_dims* sdims, const rbt_stage_ctrl* ctrl, int n_grid, int cost_structure, int i,
                        rbt_wire_layout* out) {
  if (!sdims || !ctrl || !out || i < 0 || i >= n_grid) return RBT_ERR_ARG;
  rbt_stage_layout S;
  rbt_make_stage_layout(sdims, &S);
  std::vector<rbt_wire_layout> W;
  make_wire_layouts(S, ctrl, n_grid, cost_structure, W);
  *out = W[i];
  return RBT_OK;
}

int rbt_pack_wire(const rbt_stage_dims* sdims, const rbt_stage_ctrl* ctrl, int n_grid, int cost_structure, const double* lin_host,
                  double* wire_host, long long n_ocps) {
  if (!sdims || !ctrl || n_grid <= 0 || !lin_host || !wire_host || n_ocps < 0) return RBT_ERR_ARG;
  rbt_stage_layout S;
  rbt_make_stage_layout(sdims, &S);
  std::vector<rbt_wire_layout> W;
  const long long w_ocp = make_wire_layouts(S, ctrl, n_grid, cost_structure, W);
  for (long long b = 0; b < n_ocps; ++b)
    for (int i = 0; i < n_grid; ++i)
      rbt_pack_wire_record(&W[i], lin_host + (b * n_grid + i) * S.l_stride, wire_host + b * w_ocp + W[i].ocp_off);
  return RBT_OK;
}

int rbt_riccati_solve_host(rbt_handle* h, const double* kkt_host, const double* dx0_host, double* ric_host,
                           double* dir_host, void* stream) {
  if (!h || !kkt_host || !dx0_host) return RBT_ERR_ARG;
  int rc;
  if ((rc = rbt_upload(h, RBT_BUF_KKT, kkt_host, stream))) return rc;
  if ((rc = rbt_upload(h, RBT_BUF_DX0, dx0_host, stream))) return rc;
  if ((rc = rbt_riccati_backward(h, 0, stream))) return rc;
  if ((rc = rbt_riccati_forward(h, stream))) return rc;
  if (ric_host && (rc = rbt_download(h, RBT_BUF_RIC, ric_host, stream))) return rc;
  if (dir_host && (rc = rbt_download(h, RBT_BUF_DIR, dir_host, stream))) return rc;
  return RBT_OK;
}

// ---- multi-GPU: the Newton step of every OCP on every rank ----------------------------------------------------------------
namespace {
// NCCL is reached through dlsym so that the library neither links against a particular libnccl nor fails to load without
// one: the communicator belongs to the host application, and it is the host's NCCL that must execute the collective.
typedef int (*nccl_allgather_fn)(const void*, void*, size_t, int, void*, cudaStream_t);
nccl_allgather_fn find_nccl_allgather() {
  static nccl_allgather_fn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* sym = dlsym(RTLD_DEFAULT, "ncclAllGather");  // the NCCL the host process already uses
    if (!sym) {
      void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
      if (lib) sym = dlsym(lib, "ncclAllGather");
    }
    fn = reinterpret_cast<nccl_allgather_fn>(sym);
  }
  return fn;
}

// direction records (stride d_stride) -> packed step records (the used prefix dx | du | dlmd,dgmm | dxi | dts,dts_next)
__global__ void pack_step_kernel(const double* __restrict__ dir, double* __restrict__ out, int d_stride, int step, long long n_rec) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_rec * step) return;
  const long long rec = e / step;
  const int k = int(e % step);
  out[e] = dir[rec * d_stride + k];
}
}  // namespace

int rbt_step_doubles(rbt_handle* h) { return h ? h->L.d_dts + 2 : -1; }

int rbt_pack_step(rbt_handle* h, double* packed_dev, void* stream) {
  if (!h || !packed_dev) return RBT_ERR_ARG;
  if (h->n_grid == 0) return RBT_ERR_STATE;
  RBT_CUDA(h, cudaSetDevice(h->device));
  const int step = h->L.d_dts + 2;
  const long long n_rec = (long long)h->batch * h->n_grid;
  pack_step_kernel<<<unsigned((n_rec * step + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->buf[RBT_BUF_DIR], packed_dev, h->L.d_stride, step, n_rec);
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_allgather_step(rbt_handle* h, void* nccl_comm, double* all_dev, void* stream) {
  if (!h || !nccl_comm || !all_dev) return RBT_ERR_ARG;
  if (h->n_grid == 0) return RBT_ERR_STATE;
  nccl_allgather_fn allgather = find_nccl_allgather();
  if (!allgather) {
    h->err = "[rbt_allgather_step] no NCCL in this process (ncclAllGather not found, libnccl.so.2 not loadable)";
    return RBT_ERR_STATE;
  }
  RBT_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int step = h->L.d_dts + 2;
  const long long n_rec = (long long)h->batch * h->n_grid;
  if (!h->d_step_pack) RBT_CUDA(h, dev_alloc(h->d_step_pack, size_t(h->batch) * h->n_grid_max * step));
  if (int prc = rbt_pack_step(h, h->d_step_pack.get(), stream)) return prc;
  const int rc = allgather(h->d_step_pack.get(), all_dev, size_t(n_rec) * step, /*ncclFloat64*/ 8, nccl_comm, st);
  if (rc != 0) {
    h->err = "[rbt_allgather_step] ncclAllGather failed with ncclResult_t " + std::to_string(rc);
    return RBT_ERR_CUDA;
  }
  return RBT_OK;
}

int rbt_sync(rbt_handle* h, void* stream) {
  if (!h) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaStreamSynchronize((cudaStream_t)stream));
  return RBT_OK;
}

const char* rbt_last_error(rbt_handle* h) { return h ? h->err.c_str() : "null handle"; }

long long rbt_launch_count(rbt_handle* h) { return h ? h->launches : 0; }

// ---------------------------------------------------------------------------------------------------------------
// unconstrained path
// ---------------------------------------------------------------------------------------------------------------
int rbt_unconstr_create(int nv, int N, double dt, int batch, int device, rbt_uhandle** out) {
  if (!out || nv != UINST_NV || N < 1 || batch < 1 || !(dt > 0)) return RBT_ERR_ARG;
  rbt_uhandle* h = new rbt_uhandle();
  h->nv = nv;
  h->N = N;
  h->dt = dt;
  h->batch = batch;
  h->device = device;
  h->buf.batch = batch;
  h->buf.n_grid_max = N + 1;
  rbt_make_ulayout(nv, &h->L);
  *out = h;
  RBT_CUDA(h, cudaSetDevice(device));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_KKT, h->L.k_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_RIC, h->L.r_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_FACT, h->L.f_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_DIR, h->L.d_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_DX0, h->L.nx, false));
  RBT_CUDA(h, dev_alloc(h->d_info, batch));
  RBT_CUDA(h, cudaMemset(h->d_info.get(), 0, size_t(batch) * sizeof(int)));
  return RBT_OK;
}

int rbt_unconstr_destroy(rbt_uhandle* h) {
  if (!h) return RBT_ERR_ARG;
  cudaSetDevice(h->device);
  delete h;
  return RBT_OK;
}

long long rbt_unconstr_buf_doubles(rbt_uhandle* h, int which) { return h ? h->buf.doubles(which, h->N + 1) : -1; }

double* rbt_unconstr_dev_ptr(rbt_uhandle* h, int which) { return h ? h->buf[which] : nullptr; }

int rbt_unconstr_upload(rbt_uhandle* h, int which, const double* host, void* stream) {
  if (!h || !host) return RBT_ERR_ARG;
  if (which != RBT_BUF_KKT && which != RBT_BUF_DX0 && which != RBT_BUF_LIN && which != RBT_BUF_CON && which != RBT_BUF_SOL)
    return RBT_ERR_ARG;
  if (!h->buf[which]) {
    h->err = "rbt_unconstr_upload: stage layer not set up (rbt_unconstr_stage_setup)";
    return RBT_ERR_STATE;
  }
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaMemcpyAsync(h->buf[which], host, size_t(rbt_unconstr_buf_doubles(h, which)) * 8,
                              cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return RBT_OK;
}

int rbt_unconstr_download(rbt_uhandle* h, int which, double* host, void* stream) {
  if (!h || !host || !h->buf[which]) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaMemcpyAsync(host, h->buf[which], size_t(rbt_unconstr_buf_doubles(h, which)) * 8,
                              cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return RBT_OK;
}

int rbt_unconstr_download_info(rbt_uhandle* h, int* host_flags, void* stream) {
  if (!h || !host_flags) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaMemcpyAsync(host_flags, h->d_info.get(), size_t(h->batch) * sizeof(int), cudaMemcpyDeviceToHost,
                              (cudaStream_t)stream));
  return RBT_OK;
}

static rbt::UParams make_uparams(rbt_uhandle* h, int write_fact) {
  rbt::UParams p;
  p.L = h->L;
  p.N = h->N;
  p.batch = h->batch;
  p.dt = h->dt;
  p.kkt = h->buf[RBT_BUF_KKT];
  p.ric = h->buf[RBT_BUF_RIC];
  p.fact = write_fact ? h->buf[RBT_BUF_FACT] : nullptr;
  p.dx0 = h->buf[RBT_BUF_DX0];
  p.dir = h->buf[RBT_BUF_DIR];
  p.info = h->d_info.get();
  return p;
}

int rbt_unconstr_backward(rbt_uhandle* h, int write_fact, void* stream) {
  if (!h) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (rbt::UCfg<UINST_NV>::KSTRIDE != h->L.k_stride) return RBT_ERR_STATE;
  RBT_CUDA(h, cudaMemsetAsync(h->d_info.get(), 0, size_t(h->batch) * sizeof(int), st));
  rbt::unconstr_backward_kernel<UINST_NV><<<h->batch, 32, 0, st>>>(make_uparams(h, write_fact));
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_unconstr_forward(rbt_uhandle* h, void* stream) {
  if (!h) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  rbt::unconstr_forward_kernel<UINST_NV><<<h->batch, 32, 0, (cudaStream_t)stream>>>(make_uparams(h, 0));
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_unconstr_solve_host(rbt_uhandle* h, const double* kkt_host, const double* dx0_host, double* ric_host,
                            double* dir_host, void* stream) {
  if (!h || !kkt_host || !dx0_host) return RBT_ERR_ARG;
  int rc;
  if ((rc = rbt_unconstr_upload(h, RBT_BUF_KKT, kkt_host, stream))) return rc;
  if ((rc = rbt_unconstr_upload(h, RBT_BUF_DX0, dx0_host, stream))) return rc;
  if ((rc = rbt_unconstr_backward(h, 0, stream))) return rc;
  if ((rc = rbt_unconstr_forward(h, stream))) return rc;
  if (ric_host && (rc = rbt_unconstr_download(h, RBT_BUF_RIC, ric_host, stream))) return rc;
  if (dir_host && (rc = rbt_unconstr_download(h, RBT_BUF_DIR, dir_host, stream))) return rc;
  return RBT_OK;
}

int rbt_unconstr_sync(rbt_uhandle* h, void* stream) {
  if (!h) return RBT_ERR_ARG;
  RBT_CUDA(h, cudaSetDevice(h->device));
  RBT_CUDA(h, cudaStreamSynchronize((cudaStream_t)stream));
  return RBT_OK;
}

// ---- stage layer of the unconstrained path
int rbt_unconstr_stage_layout_get(int nv, int n_box, const char* field) {
  if (nv < 1 || n_box < 0 || !field) return -1;
  rbt_ustage_layout S;
  rbt_make_ustage_layout(nv, n_box, &S);
  return rbt_ustage_layout_field(&S, field);
}

int rbt_unconstr_stage_setup(rbt_uhandle* h, const rbt_constraint_table* table) {
  if (!h || !table) return RBT_ERR_ARG;
  if (table->n_box < 0 || table->n_box > RBT_MAX_BOX_ROWS || table->n_contacts != 0 || !(table->barrier > 0) ||
      !(table->fraction_to_boundary > 0 && table->fraction_to_boundary < 1)) {
    h->err = "rbt_unconstr_stage_setup: invalid constraint table (n_box range, n_contacts must be 0, barrier > 0, 0 < fraction_to_boundary < 1)";
    return RBT_ERR_ARG;
  }
  for (int r = 0; r < table->n_box; ++r) {
    const rbt_box_row& b = table->box[r];
    if (b.var < RBT_VAR_Q || b.var > RBT_VAR_U || b.idx < 0 || b.idx >= h->nv || (b.sign != 1 && b.sign != -1)) {
      h->err = "rbt_unconstr_stage_setup: box row " + std::to_string(r) + " out of range";
      return RBT_ERR_ARG;
    }
  }
  if (h->stage_ready) {
    h->err = "rbt_unconstr_stage_setup: already set up";
    return RBT_ERR_STATE;
  }
  RBT_CUDA(h, cudaSetDevice(h->device));
  rbt_make_ustage_layout(h->nv, table->n_box, &h->S);
  h->table = *table;
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_LIN, h->S.l_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_CON, h->S.c_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_EXP, h->S.e_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_SOL, h->S.s_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_XDIR, h->S.x_stride, true));
  RBT_CUDA(h, h->buf.alloc(RBT_BUF_STEPS, 2, false));
  RBT_CUDA(h, dev_alloc(h->d_ones, size_t(h->batch) * 2));
  std::vector<double> ones(size_t(h->batch) * 2, 1.0);
  RBT_CUDA(h, cudaMemcpy(h->d_ones.get(), ones.data(), ones.size() * 8, cudaMemcpyHostToDevice));
  RBT_CUDA(h, cudaMemcpy(h->buf[RBT_BUF_STEPS], ones.data(), ones.size() * 8, cudaMemcpyHostToDevice));
  h->stage_ready = true;
  return RBT_OK;
}

static rbt::UStageParams make_ustage_params(rbt_uhandle* h) {
  rbt::UStageParams p;
  p.K = h->L;
  p.S = h->S;
  p.tab = h->table;
  p.N = h->N;
  p.batch = h->batch;
  p.dt = h->dt;
  p.lin = h->buf[RBT_BUF_LIN];
  p.con = h->buf[RBT_BUF_CON];
  p.kkt = h->buf[RBT_BUF_KKT];
  p.ex = h->buf[RBT_BUF_EXP];
  p.dir = h->buf[RBT_BUF_DIR];
  p.xd = h->buf[RBT_BUF_XDIR];
  p.sol = h->buf[RBT_BUF_SOL];
  p.steps = h->buf[RBT_BUF_STEPS];
  return p;
}

#define RBT_USTAGE_GUARD(h)                                                              \
  if (!h) return RBT_ERR_ARG;                                                            \
  if (!h->stage_ready) {                                                                 \
    h->err = "stage layer not set up: call rbt_unconstr_stage_setup first";              \
    return RBT_ERR_STATE;                                                                \
  }                                                                                      \
  RBT_CUDA(h, cudaSetDevice(h->device));                                                 \
  cudaStream_t st = (cudaStream_t)stream;

int rbt_unconstr_condense(rbt_uhandle* h, void* stream) {
  RBT_USTAGE_GUARD(h)
  const size_t total = size_t(h->batch) * (h->N + 1);
  if (rbt::UStageCfg<UINST_NV>::LSTRIDE != h->S.l_stride) return RBT_ERR_STATE;
  constexpr int W = rbt::UStageCfg<UINST_NV>::WARPS;
  rbt::ucondense_kernel<UINST_NV><<<unsigned((total + W - 1) / W), 32 * W, 0, st>>>(make_ustage_params(h));
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_unconstr_expand_and_step_sizes(rbt_uhandle* h, void* stream) {
  RBT_USTAGE_GUARD(h)
  const size_t total = size_t(h->batch) * h->N;
  RBT_CUDA(h, cudaMemcpyAsync(h->buf[RBT_BUF_STEPS], h->d_ones.get(), size_t(h->batch) * 2 * 8, cudaMemcpyDeviceToDevice, st));
  rbt::uexpand_kernel<UINST_NV><<<unsigned((total + 3) / 4), 128, 0, st>>>(make_ustage_params(h));
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_unconstr_update(rbt_uhandle* h, void* stream) {
  RBT_USTAGE_GUARD(h)
  const size_t total = size_t(h->batch) * (h->N + 1);
  rbt::uupdate_kernel<UINST_NV><<<unsigned((total + 3) / 4), 128, 0, st>>>(make_ustage_params(h));
  RBT_CUDA(h, cudaGetLastError());
  h->launches += 1;
  return RBT_OK;
}

int rbt_unconstr_iteration_host(rbt_uhandle* h, const double* lin_host, const double* con_host, const double* sol_host,
                                const double* dx0_host, double* sol_out, double* con_out, double* steps_out,
                                void* stream) {
  if (!h || !lin_host || !con_host || !sol_host || !dx0_host) return RBT_ERR_ARG;
  int rc;
  if ((rc = rbt_unconstr_upload(h, RBT_BUF_LIN, lin_host, stream))) return rc;
  if ((rc = rbt_unconstr_upload(h, RBT_BUF_CON, con_host, stream))) return rc;
  if ((rc = rbt_unconstr_upload(h, RBT_BUF_SOL, sol_host, stream))) return rc;
  if ((rc = rbt_unconstr_upload(h, RBT_BUF_DX0, dx0_host, stream))) return rc;
  if ((rc = rbt_unconstr_condense(h, stream))) return rc;
  if ((rc = rbt_unconstr_backward(h, 0, stream))) return rc;
  if ((rc = rbt_unconstr_forward(h, stream))) return rc;
  if ((rc = rbt_unconstr_expand_and_step_sizes(h, stream))) return rc;
  if ((rc = rbt_unconstr_update(h, stream))) return rc;
  if (sol_out && (rc = rbt_unconstr_download(h, RBT_BUF_SOL, sol_out, stream))) return rc;
  if (con_out && (rc = rbt_unconstr_download(h, RBT_BUF_CON, con_out, stream))) return rc;
  if (steps_out && (rc = rbt_unconstr_download(h, RBT_BUF_STEPS, steps_out, stream))) return rc;
  return RBT_OK;
}

const char* rbt_unconstr_last_error(rbt_uhandle* h) { return h ? h->err.c_str() : "null handle"; }
long long rbt_unconstr_launch_count(rbt_uhandle* h) { return h ? h->launches : 0; }

