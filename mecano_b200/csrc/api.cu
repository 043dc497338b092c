// api.cu -- the C ABI declared in include/mecano_b200.h.  Host-side plumbing only: argument checks,
// handle lifetime, kernel planning, and the chunked host<->device pipeline behind the *_host entry
// points.  There is deliberately no CPU compute path in this library: every compute entry point ends
// in a kernel launch or returns an error.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/mecano_b200.h"
#include "flatten.h"
#include "jit.h"
#include "kernels.h"
#include "ltdl_solve.cuh"
#include "specialize.h"

#define MB_STAGGER_NS_DEFAULT 0
#define MB_ABA_DISCARD_DEFAULT 1 // profiles/r04b_aba_records.md: 1.713 -> 1.696 ms, DRAM writes 2.46 -> 1.82 GB per 2^20 H37 states
#define MB_MAX_SLOTS 4
#define MB_COUNTERS 256

struct mecano_b200_handle
{
   int device = 0;
   mb::FlatTree tree;
   double *d_consts = nullptr;
   uint16_t *d_zero = nullptr; // CRBA: structurally zero entries
   uint32_t *d_yzero = nullptr; // joint-torque regressor: structurally zero rows (FlatTree::regressor_zero_rows)
   MbProgram *d_prog = nullptr; // [3] device copies of the traversal programs (warp-per-state kernels)
   std::vector<std::pair<int, int>> nonzero_runs; // CRBA: (first entry, count) runs of mass-matrix entries that are not structurally zero
   unsigned *d_counters = nullptr; // work counters of the persistent launches (kernels.cu: launch_thread_kernel): a ring of MB_COUNTERS,
   unsigned counter_seq = 0;       // a fresh one per launch, so that launches in flight on different streams never share one
   double *d_zero_row = nullptr; // one row of zeros: stands in for qd / qdd when RNEA ignores velocities / accelerations
   size_t zero_row_doubles = 0;
   double *d_scratch = nullptr; // joint efforts nobody asked for (centroidal convective term = one RNEA launch)
   size_t scratch_doubles = 0;
   double *d_ws[1 + MB_MAX_SLOTS] = {}; // ABA pass-two records: [0] device entry points, [1 + s] host-pipeline slot s
   size_t ws_doubles[1 + MB_MAX_SLOTS] = {};
   mb::SpecKernel spec[MB_NUM_ALGOS];                        // tree-specialised kernels (mecano_b200_specialize), per algorithm
   double gravity[3] = {0.0, 0.0, 0.0}; // Mecano calculators start with zero gravity until setGravitationalAcceleration
   mb::LaunchPlan plan[MB_NUM_ALGOS];
   bool fp32 = false; // mecano_b200_set_precision
   int grid_limit[MB_NUM_ALGOS] = {}; // mecano_b200_set_grid_limit: cap on the persistent grids (0 = whole device)
   int variant = MECANO_B200_VARIANT_AUTO;
   int max_children = 1, max_ndof = 1, sm_count = 148;
   int n_accel_source = 0;           // joints in ACCELERATION_SOURCE mode (mecano_b200_set_joint_source_modes)
   std::vector<std::pair<int, int>> effort_dof_runs; // (first DoF row, count) runs of DoF rows whose joints are EFFORT_SOURCE
   bool warp_ok = false;             // the body-parallel variant serves this tree (one-DoF / SixDoF joints; <= 32 bodies: a warp per state, else a team of warps)
   bool has_3dof = false;            // the tree has spherical / planar joints (generic thread-per-state kernels only)
   int64_t warp_below[MB_NUM_ALGOS] = {}; // AUTO: batches smaller than this run warp-per-state
   std::string error;
   // host pipeline (lazy)
   cudaStream_t streams[MB_MAX_SLOTS] = {};
   cudaEvent_t done[MB_MAX_SLOTS] = {};
   double *stage[MB_MAX_SLOTS] = {};
   size_t stage_doubles = 0;
   int n_slots = 3; // slots (stream + staging buffer) of the host pipeline (profiles/r04b_host_pipe.jsonl: 3 x 128 MB is 15 % faster than 2 x 64 MB)
   std::mutex mu;
};

namespace
{
std::string g_create_error;
std::mutex g_create_mu;

int fail(mecano_b200_handle *h, int code, const std::string &msg)
{
   if (h)
      h->error = msg;
   else
   {
      std::lock_guard<std::mutex> lk(g_create_mu);
      g_create_error = msg;
   }
   return code;
}

int cuda_fail(mecano_b200_handle *h, cudaError_t e, const char *what)
{
   return fail(h, (int)e > 0 ? (int)e : 1, std::string(what) + ": " + cudaGetErrorString(e));
}

#define MB_CUDA(h, call)                                  \
   do                                                     \
   {                                                      \
      cudaError_t e_ = (call);                            \
      if (e_ != cudaSuccess) return cuda_fail(h, e_, #call); \
   } while (0)

// Makes the handle's device current for the duration of an entry point and restores the caller's afterwards (a binding that
// keeps its own notion of the current device -- torch, a JVM thread pool -- must not find it changed behind its back).
struct DeviceGuard
{
   int prev = -1;
   cudaError_t err = cudaSuccess;
   explicit DeviceGuard(int device)
   {
      if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
      if (prev != device) err = cudaSetDevice(device);
      else prev = -1;
   }
   ~DeviceGuard()
   {
      if (prev >= 0) cudaSetDevice(prev);
   }
};
#define MB_ON_DEVICE(h)                                                            \
   DeviceGuard device_guard_((h)->device);                                         \
   if (device_guard_.err != cudaSuccess) return cuda_fail(h, device_guard_.err, "cudaSetDevice")

// mecano_b200_kernel_info::bytes_per_state: what one state reads and writes (MbAlgoInfo::io_*)
double bytes_per_state(int algo, double nq, double nv, double nb)
{
   const MbAlgoInfo d = mb_algo(algo);
   return 8.0 * (d.io_nq * nq + d.io_nv * nv + d.io_nv2 * nv * nv + d.io_nbnv * nb * nv);
}

int check_batch(mecano_b200_handle *h, int64_t n, int64_t ld)
{
   if (!h) return MECANO_B200_ERR_INVALID_ARGUMENT;
   if (n < 0) return fail(h, MECANO_B200_ERR_SHAPE, "n_states must be >= 0");
   if (ld < n) return fail(h, MECANO_B200_ERR_SHAPE, "ld must be >= n_states");
   return MECANO_B200_OK;
}

// optional buffers of one launch; any of them routes the call to the generic thread-per-state kernel
struct RunOpts
{
   int ws_slot = 0;                                      // ABA workspace: 0 device entry points, 1 / 2 the host-pipeline slots
   double *body_acc = nullptr, *joint_wrench = nullptr; // RNEA by-products
   const double *x2 = nullptr;                           // ABA: accelerations of the ACCELERATION_SOURCE joints
   double *cmm = nullptr, *com = nullptr;                // CRBA: centroidal momentum matrix (root frame), (mass * CoM, mass)
   double *root_wrench = nullptr;                        // RNEA: wrench at the root (root frame)
   double *cor = nullptr;                                // MB_CORIOLIS: the Coriolis matrix
   bool zero_gravity = false;
   int64_t variant_n = 0; // batch size VARIANT_AUTO decides on (0: n of this launch); the host pipelines pass the size of the whole call so
                          // that every chunk and every device slice of one call runs the same kernel (bit-identical results)
};

int run(mecano_b200_handle *h, int algo, int64_t n, int64_t ld, const double *q, const double *qd, const double *x, const double *fext,
        double *out, uint32_t flags, cudaStream_t stream, const RunOpts &opt = RunOpts())
{
   const int ws_slot = opt.ws_slot;
   double *const body_acc = opt.body_acc, *const joint_wrench = opt.joint_wrench;
   const double *x2 = opt.x2;
   if (n > (int64_t)1 << 28 || ld > (int64_t)1 << 28)
      return fail(h, MECANO_B200_ERR_TOO_LARGE, "more than 2^28 states (or ld > 2^28) in one call: split the batch");
   if (algo == MB_ABA && h->n_accel_source > 0 && !x2)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "joints in ACCELERATION_SOURCE mode need their accelerations: call mecano_b200_aba_sources");
   if (h->n_accel_source == 0)
      x2 = nullptr; // nothing reads it: the plain kernels serve the call
   const bool packed = algo == MB_CRBA && (flags & MECANO_B200_CRBA_PACKED);
   if (packed && ((flags & (MECANO_B200_CRBA_STATE_MAJOR | MECANO_B200_CRBA_ZEROS_PRESENT)) || opt.cmm || opt.com))
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "the packed mass-matrix layout does not combine with STATE_MAJOR / ZEROS_PRESENT or the centroidal by-products");
   if (h->fp32)
   {
      // the optional fp32 variant: plain calls on the thread-per-state kernels only, never a silent fp64 substitute
      if (mb_algo(algo).thread_only || packed || fext || opt.body_acc || opt.joint_wrench || x2 || opt.cmm || opt.com || opt.root_wrench || flags != 0)
         return fail(h, MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY, "the fp32 variant covers plain RNEA / ABA / CRBA calls only (no external wrenches, flags, by-products)");
      if (!h->plan[algo].fp32_ok || h->has_3dof)
         return fail(h, MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY, "the fp32 variant is compiled for the launch configuration of humanoid-sized trees of one-DoF and SixDoF joints only");
   }
   // thread- or warp-per-state: explicit choice, else by batch size (a warp per state fills the machine from a few hundred
   // states on; a thread per state needs tens of thousands but then has 10-30x the throughput)
   // calls with by-product buffers (mecano_b200_rnea_full) always run the generic thread-per-state kernel
   // (so does the packed mass-matrix layout: its row numbering follows the thread-per-state traversal)
   const bool byprod = body_acc || joint_wrench || x2 || opt.cmm || opt.com || opt.root_wrench || mb_algo(algo).thread_only || h->fp32 || packed;
   const int64_t vn = opt.variant_n > 0 ? opt.variant_n : n;
   const bool use_warp = !byprod && (h->variant == MECANO_B200_VARIANT_WARP || (h->variant == MECANO_B200_VARIANT_AUTO && h->warp_ok && vn < h->warp_below[algo]));
   if (use_warp)
   {
      if (!h->warp_ok)
         return fail(h, MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY, "the warp-per-state variant handles trees of one-DoF and SixDoF joints only");
      mb::KernelArgs wa;
      wa.q = q; wa.qd = qd; wa.x = x; wa.fext = fext; wa.out = out;
      wa.body_acc = wa.joint_wrench = nullptr;
      wa.x2 = nullptr;
      wa.cmm = wa.com = wa.root_wrench = wa.cor = nullptr;
      wa.work_counter = nullptr;
      wa.fp32 = 0;
      wa.consts = h->d_consts;
      wa.ws = nullptr;
      wa.ws_ld = 0;
      wa.zero_entries = h->d_zero;
      wa.n_zero = (algo == MB_CRBA && (flags & MECANO_B200_CRBA_ZEROS_PRESENT)) ? 0 : (int32_t)h->tree.zero_entries.size();
      wa.n = n; wa.ld = ld;
      wa.ld_qd = wa.ld_x = ld;
      wa.grav[0] = h->gravity[0]; wa.grav[1] = h->gravity[1]; wa.grav[2] = h->gravity[2];
      wa.flags = flags;
      wa.nv = h->tree.nv;
      // one lane per body: a warp per state up to 32 bodies, a team of two to four warps beyond (team_kernels.cu)
      if (h->tree.prog[algo].nb <= 32)
         MB_CUDA(h, mb::launch_warp_kernel(algo, h->d_prog + algo, wa, h->max_children, h->max_ndof, h->sm_count, stream));
      else
         MB_CUDA(h, mb::launch_team_kernel(algo, h->d_prog + algo, h->tree.prog[algo].nb, wa, h->max_children, h->max_ndof, h->sm_count, stream));
      return MECANO_B200_OK;
   }
   // the tree-specialised kernel covers the common call (no external wrenches, default flags / layout); everything else
   // runs the generic kernels
   const mb::SpecKernel &sk = h->spec[algo];
   const bool use_spec = sk.ready() && !fext && !byprod && flags == 0;
   if (algo == MB_ABA)
   {
      const size_t need = use_spec ? (size_t)sk.grid * sk.opt.block * (size_t)std::max(h->tree.prog[MB_ABA].rec_doubles, 1) : h->plan[MB_ABA].ws_doubles;
      if (h->ws_doubles[ws_slot] < need)
      {
         if (h->d_ws[ws_slot])
         {
            MB_CUDA(h, cudaStreamSynchronize(stream));
            MB_CUDA(h, cudaFree(h->d_ws[ws_slot]));
            h->d_ws[ws_slot] = nullptr;
            h->ws_doubles[ws_slot] = 0;
         }
         MB_CUDA(h, cudaMalloc(&h->d_ws[ws_slot], need * sizeof(double)));
         h->ws_doubles[ws_slot] = need;
      }
   }
   mb::KernelArgs a;
   a.q = q; a.qd = qd; a.x = x; a.fext = fext; a.out = out;
   a.body_acc = body_acc; a.joint_wrench = joint_wrench;
   a.x2 = x2;
   a.cmm = opt.cmm; a.com = opt.com; a.root_wrench = opt.root_wrench;
   a.cor = opt.cor;
   a.fp32 = h->fp32 ? 1 : 0;
   a.consts = h->d_consts;
   a.ws = h->d_ws[ws_slot];
   a.ws_ld = 0;
   a.zero_entries = h->d_zero;
   a.n_zero = (algo == MB_CRBA && (flags & (MECANO_B200_CRBA_ZEROS_PRESENT | MECANO_B200_CRBA_PACKED))) ? 0 : (int32_t)h->tree.zero_entries.size();
   if (algo == MB_REGRESSOR)
   {
      a.zero_entries = reinterpret_cast<const uint16_t *>(h->d_yzero); // (kernel_args.h: the regressor's uint32 zero rows)
      a.n_zero = (int32_t)h->tree.regressor_zero_rows.size();
   }
   a.n = n; a.ld = ld;
   a.ld_qd = a.ld_x = ld;
   if (algo == MB_RNEA && (flags & (MECANO_B200_RNEA_NO_CORIOLIS | MECANO_B200_RNEA_NO_ACCELERATIONS)))
   {
      // setConsiderCoriolisAndCentrifugalForces(false) / setConsiderJointAccelerations(false) (InverseDynamicsCalculator.java:
      // 291-306) = the same recursion with zero joint velocities / accelerations: one row of zeros with stride 0 replaces the
      // input, so the kernels carry no flag tests
      if (h->zero_row_doubles < (size_t)n)
      {
         if (h->d_zero_row)
         {
            MB_CUDA(h, cudaDeviceSynchronize());
            MB_CUDA(h, cudaFree(h->d_zero_row));
            h->d_zero_row = nullptr;
            h->zero_row_doubles = 0;
         }
         MB_CUDA(h, cudaMalloc(&h->d_zero_row, (size_t)n * sizeof(double)));
         // zeroed before any stream reads it: the host pipeline's slots launch on other streams
         MB_CUDA(h, cudaMemsetAsync(h->d_zero_row, 0, (size_t)n * sizeof(double), stream));
         MB_CUDA(h, cudaStreamSynchronize(stream));
         h->zero_row_doubles = (size_t)n;
      }
      if (flags & MECANO_B200_RNEA_NO_CORIOLIS) { a.qd = h->d_zero_row; a.ld_qd = 0; }
      if (flags & MECANO_B200_RNEA_NO_ACCELERATIONS) { a.x = h->d_zero_row; a.ld_x = 0; }
   }
   a.grav[0] = h->gravity[0]; a.grav[1] = h->gravity[1]; a.grav[2] = h->gravity[2];
   if (opt.zero_gravity)
      a.grav[0] = a.grav[1] = a.grav[2] = 0.0;
   a.flags = flags;
   if (algo == MB_ABA)
   {
      // pass three discards each record from L2 once read (gpu_ctx.cuh: rec_discard); MECANO_B200_ABA_DISCARD=0 / 1 overrides
      static const int discard = [] { const char *e = getenv("MECANO_B200_ABA_DISCARD"); return e ? atoi(e) : MB_ABA_DISCARD_DEFAULT; }();
      if (discard) a.flags |= MB_KFLAG_ABA_DISCARD;
   }
   a.nv = h->tree.nv;
   a.work_counter = (h->d_counters && !use_spec) ? h->d_counters + 2 * (h->counter_seq++ % MB_COUNTERS) : nullptr;
   {
      // MECANO_B200_STAGGER_NS overrides the start offset between the warps of a scheduler (gpu_ctx.cuh: thread_block_run)
      static const int stagger = [] { const char *e = getenv("MECANO_B200_STAGGER_NS"); return e ? atoi(e) : MB_STAGGER_NS_DEFAULT; }();
      a.stagger_ns = stagger;
   }
   if (use_spec)
   {
      const long long ntiles = (n + sk.opt.block - 1) / sk.opt.block;
      // ABA: persistent grid (workspace column per resident thread); RNEA / CRBA: one block per tile
      const unsigned grid = (algo == MB_ABA || sk.opt.tm > 0) ? (unsigned)std::min<long long>(ntiles, sk.grid) : (unsigned)ntiles;
      a.ws_ld = (long long)sk.grid * sk.opt.block;
      MB_CUDA(h, mb::spec_launch(sk, a, grid, stream));
      return MECANO_B200_OK;
   }
   if (h->grid_limit[algo] > 0 && h->grid_limit[algo] < h->plan[algo].grid)
   {
      mb::LaunchPlan p = h->plan[algo];
      p.grid = h->grid_limit[algo]; // the workspace keeps one column per thread of the full grid: enough for any smaller one
      MB_CUDA(h, mb::launch_thread_kernel(algo, h->tree.prog[algo], a, p, stream));
      return MECANO_B200_OK;
   }
   MB_CUDA(h, mb::launch_thread_kernel(algo, h->tree.prog[algo], a, h->plan[algo], stream));
   return MECANO_B200_OK;
}

// ForwardDynamicsCalculator.compute(tau, qdd_in) with per-joint source modes (ForwardDynamicsCalculator.java:508-520): passes one to
// three in the ABA kernel; pass four (:1315-1363, the efforts of the ACCELERATION_SOURCE joints from the joint wrenches) is the upward
// sweep of inverse dynamics on the accelerations just computed, i.e. one RNEA launch, after which the rows of the EFFORT_SOURCE
// joints are restored to the caller's input as getJointTauMatrix() returns them (:566-590).  opt: ws_slot and variant_n only.
int run_aba_sources(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau, const double *qdd_in,
                    const double *fext, double *qdd, double *tau_out, cudaStream_t stream, RunOpts opt)
{
   if (h->n_accel_source > 0 && !qdd_in)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer (qdd_in) with joints in ACCELERATION_SOURCE mode");
   RunOpts aba = opt;
   aba.x2 = qdd_in;
   int rc = run(h, MB_ABA, n, ld, q, qd, tau, fext, qdd, 0u, stream, aba);
   if (rc || !tau_out)
      return rc;
   const size_t row = (size_t)ld * sizeof(double);
   if (h->n_accel_source == 0)
   {
      if (tau_out != tau)
         MB_CUDA(h, cudaMemcpy2DAsync(tau_out, row, tau, row, (size_t)n * sizeof(double), (size_t)h->tree.nv, cudaMemcpyDeviceToDevice, stream));
      return MECANO_B200_OK;
   }
   if (tau_out == tau)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "tau_out must not alias tau when joints are in ACCELERATION_SOURCE mode");
   rc = run(h, MB_RNEA, n, ld, q, qd, qdd, fext, tau_out, 0u, stream, opt);
   if (rc) return rc;
   for (const auto &r : h->effort_dof_runs)
      MB_CUDA(h, cudaMemcpy2DAsync(tau_out + (size_t)r.first * ld, row, tau + (size_t)r.first * ld, row, (size_t)n * sizeof(double), (size_t)r.second,
                                   cudaMemcpyDeviceToDevice, stream));
   return MECANO_B200_OK;
}

// "rnea=512:32,aba=256:0" -> block size and TMEM stack slots of the specialised kernel of one algorithm
bool spec_cfg_from_env(int algo, mb::SpecOptions &opt)
{
   const char *e = getenv("MECANO_B200_SPEC_CFG");
   if (!e) return false;
   const char *key = algo == MB_RNEA ? "rnea=" : (algo == MB_ABA ? "aba=" : "crba=");
   const char *p = strstr(e, key);
   if (!p) return false;
   int b = 0, tm = 0, sync = 1;
   if (sscanf(p + strlen(key), "%d:%d:%d", &b, &tm, &sync) < 1 || b < 32 || b > 1024 || (b & 31)) return false;
   opt.block = b;
   opt.tm = tm;
   opt.sync_every = sync;
   return true;
}

int ensure_pipeline(mecano_b200_handle *h, size_t doubles_per_slot)
{
   for (int i = 0; i < h->n_slots; i++)
   {
      if (!h->streams[i]) MB_CUDA(h, cudaStreamCreateWithFlags(&h->streams[i], cudaStreamNonBlocking));
      if (!h->done[i]) MB_CUDA(h, cudaEventCreateWithFlags(&h->done[i], cudaEventDisableTiming));
   }
   if (doubles_per_slot > h->stage_doubles)
   {
      for (int i = 0; i < h->n_slots; i++)
      {
         if (h->stage[i]) cudaFree(h->stage[i]);
         h->stage[i] = nullptr;
      }
      h->stage_doubles = 0;
      for (int i = 0; i < h->n_slots; i++)
         MB_CUDA(h, cudaMalloc(&h->stage[i], doubles_per_slot * sizeof(double)));
      h->stage_doubles = doubles_per_slot;
   }
   return MECANO_B200_OK;
}

// rows x [s0, s0 + w) of a host matrix with leading dimension ld  <->  rows x w device matrix (ld = chunk)
cudaError_t copy_rows(double *dst, size_t dpitch, const double *src, size_t spitch, size_t w, size_t rows, cudaMemcpyKind kind, cudaStream_t s)
{
   return cudaMemcpy2DAsync(dst, dpitch * sizeof(double), src, spitch * sizeof(double), w * sizeof(double), rows, kind, s);
}

// ------------------------------------------------------------------------------------------------ jobs
// One call on one handle ("lane"), declared as matrices (entry-major, leading dimension ld) and the steps that run on them.  On
// device pointers (run_device) the job runs as one chunk of all n states on the caller's matrices.  On host pointers the pipeline
// stages each chunk in one slot: the inputs are uploaded, then each step is launched and its outputs are copied back; pointers are
// already offset to the lane's first state.
// Fixed capacities, so that a device call does not allocate: at most 5 inputs (aba_job, step_job), 3 steps (step_job) and 4
// outputs per step (aba_derivatives_job).  A value-initialised tail entry is absent; an empty launch ends the steps.
#define MB_JOB_INPUTS 5
#define MB_JOB_STEPS 3
#define MB_STEP_OUTPUTS 4
enum CopyBack
{
   COPY_ROWS,        // entry-major rows
   COPY_STATES,      // state-major: `rows` contiguous doubles per state
   COPY_NONZERO_RUNS // entry-major, the rows of h->nonzero_runs only (CRBA ZEROS_PRESENT: the host matrix already holds the zeros)
};
struct JobIn
{
   const double *host; // NULL: absent (no device rows)
   size_t rows;
};
struct JobOut
{
   double *host; // NULL: device-only scratch
   size_t rows;  // 0: absent
   CopyBack how = COPY_ROWS;
   int in = -1; // >= 0: written in place into the device rows of that input
};
// what a step's launch sees: the device rows (NULL for an absent matrix) of every input and of the step's outputs, the width w,
// their leading dimension ld (the chunk in the pipeline) and the stream and options (ws_slot, variant_n)
struct Chunk
{
   mecano_b200_handle *h;
   const double *in[MB_JOB_INPUTS];
   double *out[MB_STEP_OUTPUTS];
   int64_t w = 0, ld = 0;
   cudaStream_t stream = nullptr;
   RunOpts opt;
};
struct JobStep
{
   std::function<int(const Chunk &)> launch; // captures a flag word, a frame, dt or a bool at most: stored inline, no allocation
   JobOut out[MB_STEP_OUTPUTS];
};
struct Job
{
   int64_t n = 0, ld = 0;
   JobIn in[MB_JOB_INPUTS];
   JobStep steps[MB_JOB_STEPS];
   int64_t variant_n = 0; // size of the whole call (all lanes)
   // staging per slot (r06ze: 229 ms per dense 2^20-state step against 239 ms with 128 MB, 231 ms with 512 MB)
   double budget_mb = 256.0;
   // pipeline state
   size_t chunk = 0;
   int64_t s0 = 0;
   int slot = 0;
};

// chunk size and staging buffers (arguments are checked by the job builders).  n_slots slots per handle, each with its own stream:
// H2D of chunk k+1 overlaps the kernels and the D2H of chunk k.
int host_begin(mecano_b200_handle *h, Job &j)
{
   if (j.n == 0) return MECANO_B200_OK;
   size_t rows = 0; // device rows per state of one slot
   for (const JobIn &i : j.in)
      rows += i.host ? i.rows : 0;
   for (const JobStep &s : j.steps)
      for (const JobOut &o : s.out)
         rows += o.in < 0 ? o.rows : 0;
   // chunk: the job's budget of rows per slot (MECANO_B200_HOST_CHUNK_MB overrides every job's), multiple of 256, at least 256 states
   // (no more: a wide job -- the regressor, a dense mass matrix of nv > 90 -- would otherwise make every slot far larger than the budget)
   static const double env_mb = [] { const char *e = getenv("MECANO_B200_HOST_CHUNK_MB"); const double v = e ? atof(e) : 0.0; return v >= 1.0 ? v : 0.0; }();
   size_t chunk = (size_t)((env_mb > 0.0 ? env_mb : j.budget_mb) * 1024 * 1024 / 8 / (double)rows);
   chunk = std::max<size_t>(256, chunk & ~(size_t)255);
   chunk = std::min<size_t>(chunk, ((size_t)j.n + 255) & ~(size_t)255);
   j.chunk = chunk;
   j.s0 = 0;
   j.slot = 0;
   MB_ON_DEVICE(h);
   return ensure_pipeline(h, rows * chunk);
}

// issues the next chunk of the job (H2D, then each step's kernels and D2H, on the slot's stream); asynchronous with pinned host memory
int host_issue_chunk(mecano_b200_handle *h, Job &j)
{
   if (j.s0 >= j.n) return MECANO_B200_OK;
   MB_ON_DEVICE(h);
   const size_t chunk = j.chunk, ld = (size_t)j.ld;
   const int64_t s0 = j.s0;
   const size_t w = (size_t)std::min<int64_t>((int64_t)chunk, j.n - s0);
   const int slot = j.slot;
   cudaStream_t st = h->streams[slot];
   j.s0 += (int64_t)chunk;
   j.slot = (slot + 1) % h->n_slots;
   // a slot is reused every n_slots chunks: stream order already serialises it
   double *p = h->stage[slot];
   double *in[MB_JOB_INPUTS] = {}; // the inputs' rows, also written by in-place outputs
   Chunk c{h, {}, {}, (int64_t)w, (int64_t)chunk, st};
   c.opt.ws_slot = 1 + slot;
   c.opt.variant_n = j.variant_n > 0 ? j.variant_n : j.n;
   for (int k = 0; k < MB_JOB_INPUTS; k++)
   {
      const JobIn &i = j.in[k];
      if (!i.host) continue;
      c.in[k] = in[k] = p;
      MB_CUDA(h, copy_rows(p, chunk, i.host + s0, ld, w, i.rows, cudaMemcpyHostToDevice, st));
      p += i.rows * chunk;
   }
   for (const JobStep &s : j.steps)
   {
      if (!s.launch) break;
      for (int k = 0; k < MB_STEP_OUTPUTS; k++)
      {
         const JobOut &o = s.out[k];
         c.out[k] = o.in >= 0 ? in[o.in] : (o.rows ? p : nullptr);
         if (o.in < 0) p += o.rows * chunk;
      }
      const int rc = s.launch(c);
      if (rc) return rc;
      for (int k = 0; k < MB_STEP_OUTPUTS; k++)
      {
         const JobOut &o = s.out[k];
         const double *d = c.out[k];
         if (!o.host || !o.rows) continue;
         if (o.how == COPY_STATES)
            MB_CUDA(h, cudaMemcpyAsync(o.host + (size_t)s0 * o.rows, d, w * o.rows * sizeof(double), cudaMemcpyDeviceToHost, st));
         else if (o.how == COPY_NONZERO_RUNS)
         {
            for (const auto &run : h->nonzero_runs)
               MB_CUDA(h, copy_rows(o.host + (size_t)run.first * ld + s0, ld, d + (size_t)run.first * chunk, chunk, w, (size_t)run.second, cudaMemcpyDeviceToHost, st));
         }
         else
            MB_CUDA(h, copy_rows(o.host + s0, ld, d, chunk, w, o.rows, cudaMemcpyDeviceToHost, st));
      }
   }
   return MECANO_B200_OK;
}

int host_finish(mecano_b200_handle *h)
{
   MB_ON_DEVICE(h);
   for (int i = 0; i < h->n_slots; i++)
      if (h->streams[i]) MB_CUDA(h, cudaStreamSynchronize(h->streams[i]));
   return MECANO_B200_OK;
}

// Runs one job per lane: the chunks of all lanes are issued round-robin from the calling thread (everything is asynchronous
// with pinned host memory), then every lane is synchronised once.  lanes.size() == 1 is the single-device host call.
int run_host_lanes(const std::vector<mecano_b200_handle *> &lanes, std::vector<Job> &jobs, int *failed_lane)
{
   int rc = MECANO_B200_OK;
   size_t started = 0;
   *failed_lane = 0;
   // a listed handle is locked for the whole call (handles are distinct objects even when they share a device)
   for (; started < lanes.size(); started++)
   {
      lanes[started]->mu.lock();
      rc = host_begin(lanes[started], jobs[started]);
      if (rc) { *failed_lane = (int)started; started++; break; }
   }
   bool pending = rc == MECANO_B200_OK;
   while (pending && rc == MECANO_B200_OK)
   {
      pending = false;
      for (size_t i = 0; i < lanes.size() && rc == MECANO_B200_OK; i++)
      {
         if (jobs[i].s0 >= jobs[i].n) continue;
         rc = host_issue_chunk(lanes[i], jobs[i]);
         if (rc) *failed_lane = (int)i;
         pending = pending || jobs[i].s0 < jobs[i].n;
      }
   }
   // always drain what was issued, also after an error: the staging buffers and the caller's matrices are in flight
   for (size_t i = 0; i < started; i++)
   {
      if (jobs[i].n > 0 && lanes[i]->streams[0])
      {
         const int rf = host_finish(lanes[i]);
         if (rf && !rc) { rc = rf; *failed_lane = (int)i; }
      }
      lanes[i]->mu.unlock();
   }
   return rc;
}

int run_host(mecano_b200_handle *h, const Job &job)
{
   std::vector<mecano_b200_handle *> lanes(1, h);
   std::vector<Job> jobs(1, job);
   int failed = 0;
   return run_host_lanes(lanes, jobs, &failed);
}

// Runs a job on the caller's device pointers: one chunk of all n states, no staging, with the options of a device entry point
// (ABA workspace slot 0, VARIANT_AUTO on n).  Every input and output is the caller's matrix, except device-only scratch, which lives
// in h->d_scratch.  Like every device entry point it takes no lock.
int run_device(mecano_b200_handle *h, const Job &j, void *stream)
{
   if (j.n == 0) return MECANO_B200_OK;
   MB_ON_DEVICE(h);
   const size_t ld = (size_t)j.ld;
   size_t rows = 0; // scratch rows
   for (const JobStep &s : j.steps)
      for (const JobOut &o : s.out)
         rows += o.host ? 0 : o.rows;
   if (h->scratch_doubles < rows * ld)
   {
      if (h->d_scratch)
      {
         MB_CUDA(h, cudaDeviceSynchronize());
         MB_CUDA(h, cudaFree(h->d_scratch));
         h->d_scratch = nullptr;
         h->scratch_doubles = 0;
      }
      MB_CUDA(h, cudaMalloc(&h->d_scratch, rows * ld * sizeof(double)));
      h->scratch_doubles = rows * ld;
   }
   Chunk c{h, {}, {}, j.n, j.ld, (cudaStream_t)stream};
   for (int k = 0; k < MB_JOB_INPUTS; k++)
      c.in[k] = j.in[k].host;
   double *p = h->d_scratch;
   for (const JobStep &s : j.steps)
   {
      if (!s.launch) break;
      for (int k = 0; k < MB_STEP_OUTPUTS; k++)
      {
         const JobOut &o = s.out[k];
         c.out[k] = !o.rows ? nullptr : o.host ? o.host : p;
         if (!o.host) p += o.rows * ld;
      }
      const int rc = s.launch(c);
      if (rc) return rc;
   }
   return MECANO_B200_OK;
}

// refusals shared by several calls
bool wrench_ranks_below_nb(const MbProgram &P)
{
   for (int i = 0; i < P.nb; i++)
      if (P.body[i].ext_index >= P.nb) return false;
   return true;
}

// a by-product kernel that did not fit the tree at mecano_b200_create (plan block 0)
int refuse_unfit(mecano_b200_handle *h, const char *kernel)
{
   return fail(h, MECANO_B200_ERR_TOO_LARGE, std::string("tree exceeds the per-state work areas of the ") + kernel + " kernel (branch nesting / depth too large)");
}

// subject: "<result> is" / "<results> are"
int refuse_fp32(mecano_b200_handle *h, const char *subject)
{
   return fail(h, MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY, std::string("the ") + subject + " computed in fp64 only (mecano_b200_set_precision)");
}

// The job of each call, shared by its device and host entry points (and by the multi-device calls): argument checks in the order
// the entry points report them (an empty batch gives an empty job), then the job.
int rnea_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, const double *fext, double *tau,
             double *body_acc, double *joint_wrench, uint32_t flags, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc || n == 0) return rc;
   if (!q || !qd || !qdd || !tau) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   const size_t nq = h->tree.nq, nv = h->tree.nv, nw = 6 * (size_t)h->tree.nb;
   j = Job{n, ld, {{q, nq}, {qd, nv}, {qdd, nv}, {fext, nw}}};
   j.steps[0] = {[flags](const Chunk &c) {
      RunOpts opt = c.opt;
      opt.body_acc = c.out[1];
      opt.joint_wrench = c.out[2];
      return run(c.h, MB_RNEA, c.w, c.ld, c.in[0], c.in[1], c.in[2], c.in[3], c.out[0], flags, c.stream, opt);
   }, {{tau, nv}, {body_acc, body_acc ? nw : 0}, {joint_wrench, joint_wrench ? nw : 0}}};
   return MECANO_B200_OK;
}

// sources: mecano_b200_aba_sources[_host] (qdd_in, tau_out; no flags)
int aba_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau, const double *qdd_in,
            const double *fext, double *qdd, double *tau_out, uint32_t flags, bool sources, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc || n == 0) return rc;
   if (!q || !qd || !tau || !qdd) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   const size_t nq = h->tree.nq, nv = h->tree.nv;
   j = Job{n, ld, {{q, nq}, {qd, nv}, {tau, nv}, {fext, 6 * (size_t)h->tree.nb}, {qdd_in, nv}}};
   j.steps[0] = {[flags, sources](const Chunk &c) {
      if (sources) return run_aba_sources(c.h, c.w, c.ld, c.in[0], c.in[1], c.in[2], c.in[4], c.in[3], c.out[0], c.out[1], c.stream, c.opt);
      return run(c.h, MB_ABA, c.w, c.ld, c.in[0], c.in[1], c.in[2], c.in[3], c.out[0], flags, c.stream, c.opt);
   }, {{qdd, nv}, {tau_out, tau_out ? nv : 0}}};
   return MECANO_B200_OK;
}

// mecano_b200_step_host: inputs q, qd, qdd_in, tau_in, fext; steps RNEA -> tau_out, ABA -> qdd_out, CRBA -> M, each one present
// when its buffers are (M alone: mecano_b200_crba_host)
int step_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd_in, const double *tau_in,
             const double *fext, double *tau_out, double *qdd_out, double *M, uint32_t layout, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc || n == 0) return rc;
   const bool rnea = qdd_in || tau_out, aba = tau_in || qdd_out;
   if (!q || ((rnea || aba) && !qd) || (rnea && (!qdd_in || !tau_out)) || (aba && (!tau_in || !qdd_out)) || (!rnea && !aba && !M))
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (aba && h->n_accel_source > 0)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "joints in ACCELERATION_SOURCE mode need their accelerations: call mecano_b200_aba_sources_host");
   if ((layout & MECANO_B200_CRBA_PACKED) && (layout & (MECANO_B200_CRBA_STATE_MAJOR | MECANO_B200_CRBA_ZEROS_PRESENT)))
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "the packed mass-matrix layout does not combine with STATE_MAJOR / ZEROS_PRESENT");
   // state-major: the whole per-state block is copied back from the staging buffer, which other calls on this handle reuse, so
   // the kernel must write the structural zeros there every time (the transfer saving of ZEROS_PRESENT is entry-major only)
   if (layout & MECANO_B200_CRBA_STATE_MAJOR)
      layout &= ~MECANO_B200_CRBA_ZEROS_PRESENT;
   const size_t nq = h->tree.nq, nv = h->tree.nv;
   j = Job{n, ld, {{q, nq}, {rnea || aba ? qd : nullptr, nv}, {qdd_in, nv}, {tau_in, nv}, {fext, 6 * (size_t)h->tree.nb}}};
   int s = 0;
   if (rnea)
      j.steps[s++] = {[](const Chunk &c) { return run(c.h, MB_RNEA, c.w, c.ld, c.in[0], c.in[1], c.in[2], c.in[4], c.out[0], 0u, c.stream, c.opt); },
                      {{tau_out, nv}}};
   if (aba)
      j.steps[s++] = {[](const Chunk &c) { return run(c.h, MB_ABA, c.w, c.ld, c.in[0], c.in[1], c.in[3], c.in[4], c.out[0], 0u, c.stream, c.opt); },
                      {{qdd_out, nv}}};
   if (M)
   {
      const CopyBack how = (layout & MECANO_B200_CRBA_STATE_MAJOR) ? COPY_STATES : (layout & MECANO_B200_CRBA_ZEROS_PRESENT) ? COPY_NONZERO_RUNS : COPY_ROWS;
      j.steps[s++] = {[layout](const Chunk &c) { return run(c.h, MB_CRBA, c.w, c.ld, c.in[0], nullptr, nullptr, nullptr, c.out[0], layout, c.stream, c.opt); },
                      {{M, (layout & MECANO_B200_CRBA_PACKED) ? h->tree.packed_row.size() : nv * nv, how}}};
   }
   return MECANO_B200_OK;
}

// mecano_b200_crba_centroidal, and with com_only (M = cmm = NULL) mecano_b200_center_of_mass.  The latter is the by-product CRBA
// kernel launched without a matrix: it keeps the composite-inertia recursion and drops the unit momenta, their ancestor walks and
// every matrix store (crba.cuh: com_only) -- the same arithmetic, hence the same bits, as the com rows of the former.
int centroidal_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, double *M, double *cmm, double *com, int frame, bool com_only,
                   Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc || n == 0) return rc;
   if (!q || (!com_only && (!M || !cmm)) || !com) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (frame != MECANO_B200_FRAME_WORLD && frame != MECANO_B200_FRAME_CENTER_OF_MASS)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "unknown centroidal momentum frame");
   const size_t nv = h->tree.nv;
   j = Job{n, ld, {{q, (size_t)h->tree.nq}}};
   j.steps[0] = {[frame](const Chunk &c) {
      double *const cmm = c.out[1], *const com = c.out[2];
      // the kernel sums (mass * CoM, mass) over the children of the root body into the com rows
      MB_CUDA(c.h, cudaMemset2DAsync(com, (size_t)c.ld * sizeof(double), 0, (size_t)c.w * sizeof(double), 4, c.stream));
      RunOpts opt = c.opt;
      opt.cmm = cmm;
      opt.com = com;
      const int rc = run(c.h, MB_CRBA, c.w, c.ld, c.in[0], nullptr, nullptr, nullptr, c.out[0], MECANO_B200_CRBA_ENTRY_MAJOR, c.stream, opt);
      if (rc) return rc;
      mb::CentroidalArgs ca;
      ca.cols = cmm; ca.com = com; ca.n = c.w; ca.ld = c.ld; ca.ncols = cmm ? c.h->tree.nv : 0;
      ca.normalize_com = 1;
      ca.shift = frame == MECANO_B200_FRAME_CENTER_OF_MASS;
      MB_CUDA(c.h, mb::launch_centroidal_finish(ca, c.stream));
      return MECANO_B200_OK;
   }, {{M, com_only ? 0 : nv * nv}, {cmm, com_only ? 0 : 6 * nv}, {com, 4}}};
   return MECANO_B200_OK;
}

// mecano_b200_centroidal_convective_term; the joint efforts nobody reads are device-only scratch
int convective_term_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *com, double *out, int frame,
                        Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc || n == 0) return rc;
   if (!q || !qd || !out) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (frame != MECANO_B200_FRAME_WORLD && frame != MECANO_B200_FRAME_CENTER_OF_MASS)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "unknown centroidal momentum frame");
   if (frame == MECANO_B200_FRAME_CENTER_OF_MASS && !com)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "the centre-of-mass frame needs the com rows of mecano_b200_crba_centroidal");
   const size_t nv = h->tree.nv;
   j = Job{n, ld, {{q, (size_t)h->tree.nq}, {qd, nv}, {com, 4}}};
   j.steps[0] = {[frame](const Chunk &c) {
      // :811-839: the net wrench of every body under zero joint accelerations and no gravity, summed in the centroidal frame = the
      // wrench at the root of inverse dynamics run that way
      MB_CUDA(c.h, cudaMemset2DAsync(c.out[0], (size_t)c.ld * sizeof(double), 0, (size_t)c.w * sizeof(double), 6, c.stream));
      RunOpts opt = c.opt;
      opt.root_wrench = c.out[0];
      opt.zero_gravity = true;
      const int rc = run(c.h, MB_RNEA, c.w, c.ld, c.in[0], c.in[1], c.in[1], nullptr, c.out[1], MECANO_B200_RNEA_NO_ACCELERATIONS, c.stream, opt);
      if (rc) return rc;
      if (frame == MECANO_B200_FRAME_CENTER_OF_MASS)
      {
         mb::CentroidalArgs ca;
         ca.cols = c.out[0]; ca.com = const_cast<double *>(c.in[2]); ca.n = c.w; ca.ld = c.ld; ca.ncols = 1; // (com is read only: normalize_com = 0)
         ca.normalize_com = 0;
         ca.shift = 1;
         MB_CUDA(c.h, mb::launch_centroidal_finish(ca, c.stream));
      }
      return MECANO_B200_OK;
   }, {{out, 6}, {nullptr, nv}}};
   return MECANO_B200_OK;
}

int coriolis_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, double *M, double *C, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc || n == 0) return rc;
   if (!q || !qd || !M || !C) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (h->plan[MB_CORIOLIS].block == 0) return refuse_unfit(h, "Coriolis-matrix");
   const size_t nv = h->tree.nv;
   j = Job{n, ld, {{q, (size_t)h->tree.nq}, {qd, nv}}};
   j.steps[0] = {[](const Chunk &c) {
      RunOpts opt = c.opt;
      opt.cor = c.out[1];
      return run(c.h, MB_CORIOLIS, c.w, c.ld, c.in[0], c.in[1], c.in[1], nullptr, c.out[0], 0u, c.stream, opt);
   }, {{M, nv * nv}, {C, nv * nv}}};
   return MECANO_B200_OK;
}

int regressor_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, double *Y, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc) return rc;
   if (h->fp32) return refuse_fp32(h, "joint-torque regressor is");
   if (!wrench_ranks_below_nb(h->tree.prog[MB_REGRESSOR]))
      return fail(h, MECANO_B200_ERR_SHAPE, "joint-torque regressor: wrench_index ranks must be below n_bodies (one ten-column block per body)");
   if (h->plan[MB_REGRESSOR].block == 0) return refuse_unfit(h, "joint-torque regressor");
   if (n == 0) return MECANO_B200_OK;
   if (!q || !qd || !qdd || !Y) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   const size_t nv = h->tree.nv;
   j = Job{n, ld, {{q, (size_t)h->tree.nq}, {qd, nv}, {qdd, nv}}};
   j.steps[0] = {[](const Chunk &c) { return run(c.h, MB_REGRESSOR, c.w, c.ld, c.in[0], c.in[1], c.in[2], nullptr, c.out[0], 0u, c.stream, c.opt); },
                 {{Y, nv * 10 * (size_t)h->tree.nb}}};
   return MECANO_B200_OK;
}

int gravity_gradient_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *fext, double *tau, double *G, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc) return rc;
   if (h->fp32) return refuse_fp32(h, "gravity gradient is");
   if (h->plan[MB_GRAVITY_GRADIENT].block == 0) return refuse_unfit(h, "gravity-gradient");
   if (n > 0 && (!q || !tau || !G)) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (fext && !wrench_ranks_below_nb(h->tree.prog[MB_GRAVITY_GRADIENT]))
      return fail(h, MECANO_B200_ERR_SHAPE, "gravity gradient: with external wrenches the wrench_index ranks must be below n_bodies (fext has 6 n_bodies rows)");
   if (n == 0) return MECANO_B200_OK;
   const size_t nv = h->tree.nv;
   j = Job{n, ld, {{q, (size_t)h->tree.nq}, {fext, 6 * (size_t)h->tree.nb}}};
   j.steps[0] = {[](const Chunk &c) {
      RunOpts opt = c.opt;
      opt.cor = c.out[0]; // (kernel_args.h: the joint efforts travel in `cor`, G in `out`)
      return run(c.h, MB_GRAVITY_GRADIENT, c.w, c.ld, c.in[0], nullptr, nullptr, c.in[1], c.out[1], 0u, c.stream, opt);
   }, {{tau, nv}, {G, nv * nv}}};
   return MECANO_B200_OK;
}

int rnea_derivatives_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, const double *fext,
                         double *tau, double *dq, double *dqd, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc) return rc;
   if (h->fp32) return refuse_fp32(h, "inverse-dynamics derivatives are");
   if (h->plan[MB_RNEA_DERIVATIVES].block == 0) return refuse_unfit(h, "inverse-dynamics derivatives");
   if (n > 0 && (!q || !qd || !qdd || !tau || !dq || !dqd)) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (fext && !wrench_ranks_below_nb(h->tree.prog[MB_RNEA_DERIVATIVES]))
      return fail(h, MECANO_B200_ERR_SHAPE, "inverse-dynamics derivatives: with external wrenches the wrench_index ranks must be below n_bodies (fext has 6 n_bodies rows)");
   if (n == 0) return MECANO_B200_OK;
   const size_t nv = h->tree.nv;
   j = Job{n, ld, {{q, (size_t)h->tree.nq}, {qd, nv}, {qdd, nv}, {fext, 6 * (size_t)h->tree.nb}}};
   j.steps[0] = {[](const Chunk &c) {
      RunOpts opt = c.opt;
      opt.root_wrench = c.out[0]; // (kernel_args.h: d tau / dq travels in `out`, d tau / dqd in `cor`,
      opt.cor = c.out[2];         //  the joint efforts in `root_wrench`)
      return run(c.h, MB_RNEA_DERIVATIVES, c.w, c.ld, c.in[0], c.in[1], c.in[2], c.in[3], c.out[1], 0u, c.stream, opt);
   }, {{tau, nv}, {dq, nv * nv}, {dqd, nv * nv}}};
   return MECANO_B200_OK;
}

// mecano_b200_aba_derivatives: the refusals of ABA and of the inverse-dynamics derivatives, whose kernels it reuses, then one step of
// four launches in stream order: ABA (qdd), the inverse-dynamics derivatives at that qdd (into dq and dqd, their joint efforts into
// the first rows of minv, which nobody reads), CRBA (M into minv) and the L^T D L solve (ltdl_solve.cuh), which turns minv into M^-1
// and dq, dqd into -M^-1 dq, -M^-1 dqd in place.  One step, so that in the pipeline the three matrices pass from launch to launch in
// the slot's rows and are copied back once, after the solve; the options are the call's (ws_slot, variant_n), so that qdd is what
// mecano_b200_aba computes.
int aba_derivatives_job(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau, const double *fext,
                        double *qdd, double *dq, double *dqd, double *minv, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc) return rc;
   if (h->fp32) return refuse_fp32(h, "forward-dynamics derivatives are");
   if (h->n_accel_source > 0)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "the forward-dynamics derivatives need every joint in EFFORT_SOURCE mode (mecano_b200_set_joint_source_modes)");
   if (h->plan[MB_RNEA_DERIVATIVES].block == 0) return refuse_unfit(h, "inverse-dynamics derivatives");
   if (n > 0 && (!q || !qd || !tau || !qdd || !dq || !dqd || !minv)) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (fext && !wrench_ranks_below_nb(h->tree.prog[MB_RNEA_DERIVATIVES]))
      return fail(h, MECANO_B200_ERR_SHAPE, "forward-dynamics derivatives: with external wrenches the wrench_index ranks must be below n_bodies (fext has 6 n_bodies rows)");
   if (n == 0) return MECANO_B200_OK;
   const size_t nv = h->tree.nv;
   j = Job{n, ld, {{q, (size_t)h->tree.nq}, {qd, nv}, {tau, nv}, {fext, 6 * (size_t)h->tree.nb}}};
   j.steps[0] = {[](const Chunk &c) {
      double *const qdd = c.out[0], *const dq = c.out[1], *const dqd = c.out[2], *const minv = c.out[3];
      int rc = run(c.h, MB_ABA, c.w, c.ld, c.in[0], c.in[1], c.in[2], c.in[3], qdd, 0u, c.stream, c.opt);
      if (rc) return rc;
      RunOpts rd = c.opt;
      rd.cor = dqd;
      rd.root_wrench = minv;
      if ((rc = run(c.h, MB_RNEA_DERIVATIVES, c.w, c.ld, c.in[0], c.in[1], qdd, c.in[3], dq, 0u, c.stream, rd))) return rc;
      if ((rc = run(c.h, MB_CRBA, c.w, c.ld, c.in[0], nullptr, nullptr, nullptr, minv, MECANO_B200_CRBA_ENTRY_MAJOR, c.stream, c.opt))) return rc;
      mb::LtdlTree t;
      t.nv = c.h->tree.nv;
      std::copy(c.h->tree.ltdl_dof.begin(), c.h->tree.ltdl_dof.end(), t.dof);
      std::copy(c.h->tree.ltdl_parent.begin(), c.h->tree.ltdl_parent.end(), t.lam);
      mb::LtdlArgs a;
      a.minv = minv; a.dq = dq; a.dqd = dqd;
      a.n = c.w; a.ld = c.ld;
      MB_CUDA(c.h, mb::launch_ltdl_solve(t, a, c.stream));
      return MECANO_B200_OK;
   }, {{qdd, nv}, {dq, nv * nv}, {dqd, nv * nv}, {minv, nv * nv}}};
   return MECANO_B200_OK;
}

// mecano_b200_integrate: q, qd and qdd are updated in place, so the step writes them through its outputs
int integrate_job(mecano_b200_handle *h, int64_t n, int64_t ld, double dt, double *q, double *qd, double *qdd, Job &j)
{
   int rc = check_batch(h, n, ld);
   if (rc || n == 0) return rc;
   if (!q || !qd || !qdd) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   if (!(dt == dt)) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "dt is NaN");
   const size_t nq = h->tree.nq, nv = h->tree.nv;
   j = Job{n, ld, {{q, nq}, {qd, nv}, {qdd, nv}}};
   j.budget_mb = 64.0; // 2^20 H37 states on a B200 (1000 W), pinned: 22 ms per call against 24 ms with 256 MB per slot; pageable 148 against 153 ms
   j.steps[0] = {[dt](const Chunk &c) {
      mb::IntegrateJoints J;
      const MbProgram &P = c.h->tree.prog[MB_RNEA];
      J.nb = P.nb;
      for (int i = 0; i < P.nb; i++)
      {
         J.cfg[i] = (uint16_t)P.body[i].cfg_off;
         J.dof[i] = (uint16_t)P.body[i].dof_off;
         J.type[i] = (uint8_t)P.body[i].jtype;
         J.sub[i] = (uint8_t)P.body[i].sub;
      }
      mb::IntegrateArgs a;
      a.q = c.out[0]; a.qd = c.out[1]; a.qdd = c.out[2];
      a.n = c.w; a.ld = c.ld;
      a.dt = dt;
      MB_CUDA(c.h, mb::launch_integrate_kernel(J, a, c.h->sm_count, c.stream));
      return MECANO_B200_OK;
   }, {{q, nq, COPY_ROWS, 0}, {qd, nv, COPY_ROWS, 1}, {qdd, nv, COPY_ROWS, 2}}};
   return MECANO_B200_OK;
}
} // namespace

extern "C" {
#pragma GCC visibility push(default)

int mecano_b200_version(void) { return MECANO_B200_VERSION; }

int mecano_b200_device_count(void)
{
   int n = 0;
   if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
   return n;
}

int mecano_b200_create(const mecano_b200_tree_desc *desc, int device, mecano_b200_handle **out)
{
   if (!out) return fail(nullptr, MECANO_B200_ERR_INVALID_ARGUMENT, "out handle pointer is NULL");
   *out = nullptr;
   mecano_b200_handle *h = new mecano_b200_handle();
   std::string err;
   int rc = mb::flatten_tree(desc, h->tree, err);
   if (rc != MECANO_B200_OK)
   {
      delete h;
      return fail(nullptr, rc, err);
   }
   int ndev = 0;
   cudaError_t e = cudaGetDeviceCount(&ndev);
   if (e != cudaSuccess || ndev == 0)
   {
      delete h;
      return fail(nullptr, MECANO_B200_ERR_NO_DEVICE,
                  std::string("no CUDA device available (this engine has no CPU fallback)") + (e != cudaSuccess ? std::string(": ") + cudaGetErrorString(e) : ""));
   }
   if (device < 0 || device >= ndev)
   {
      delete h;
      return fail(nullptr, MECANO_B200_ERR_INVALID_ARGUMENT, "device index out of range");
   }
   h->device = device;
   if (const char *es = getenv("MECANO_B200_HOST_SLOTS"))
      h->n_slots = std::min(MB_MAX_SLOTS, std::max(1, atoi(es)));
   auto bail = [&](cudaError_t ce, const char *what) {
      mecano_b200_destroy(h);
      return fail(nullptr, (int)ce, std::string(what) + ": " + cudaGetErrorString(ce));
   };
   DeviceGuard device_guard_(device);
   if ((e = device_guard_.err) != cudaSuccess) return bail(e, "cudaSetDevice");
   const size_t bytes = h->tree.consts.size() * sizeof(double);
   if ((e = cudaMalloc(&h->d_consts, bytes)) != cudaSuccess) return bail(e, "cudaMalloc(consts)");
   if ((e = cudaMalloc(&h->d_counters, 2 * sizeof(unsigned) * MB_COUNTERS)) != cudaSuccess) return bail(e, "cudaMalloc(counters)");
   if ((e = cudaMemset(h->d_counters, 0, 2 * sizeof(unsigned) * MB_COUNTERS)) != cudaSuccess) return bail(e, "cudaMemset(counters)");
   if ((e = cudaMemcpy(h->d_consts, h->tree.consts.data(), bytes, cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "cudaMemcpy(consts)");
   {
      std::vector<char> isz((size_t)h->tree.nv * h->tree.nv, 0);
      for (uint16_t e : h->tree.zero_entries)
         isz[e] = 1;
      for (int e = 0; e < (int)isz.size(); e++)
      {
         if (isz[(size_t)e])
            continue;
         if (!h->nonzero_runs.empty() && h->nonzero_runs.back().first + h->nonzero_runs.back().second == e)
            h->nonzero_runs.back().second++;
         else
            h->nonzero_runs.emplace_back(e, 1);
      }
   }
   if (!h->tree.zero_entries.empty())
   {
      const size_t zb = h->tree.zero_entries.size() * sizeof(uint16_t);
      if ((e = cudaMalloc(&h->d_zero, zb)) != cudaSuccess) return bail(e, "cudaMalloc(zero entries)");
      if ((e = cudaMemcpy(h->d_zero, h->tree.zero_entries.data(), zb, cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "cudaMemcpy(zero entries)");
   }
   if (!h->tree.regressor_zero_rows.empty())
   {
      const size_t zb = h->tree.regressor_zero_rows.size() * sizeof(uint32_t);
      if ((e = cudaMalloc(&h->d_yzero, zb)) != cudaSuccess) return bail(e, "cudaMalloc(regressor zero rows)");
      if ((e = cudaMemcpy(h->d_yzero, h->tree.regressor_zero_rows.data(), zb, cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "cudaMemcpy(regressor zero rows)");
   }
   for (int algo = 0; algo < MB_NUM_ALGOS; algo++)
   {
      bool fits = false;
      if ((e = mb::plan_thread_kernel(algo, h->tree.prog[algo], false, h->plan[algo], &fits)) != cudaSuccess) return bail(e, "kernel planning");
      if (!fits && mb_algo(algo).thread_only)
      {
         h->plan[algo].block = 0; // a by-product kernel alone does not fit: its entry point reports it, everything else works
         continue;
      }
      if (!fits)
      {
         mecano_b200_destroy(h);
         return fail(nullptr, MECANO_B200_ERR_TOO_LARGE, "tree exceeds the compiled per-state work areas (branch nesting / depth too large)");
      }
   }
   {
      const MbProgram &P = h->tree.prog[MB_RNEA];
      std::vector<int> nchild(P.nb, 0);
      for (int i = 0; i < P.nb; i++)
      {
         if (P.body[i].parent >= 0) nchild[P.body[i].parent]++;
         h->max_ndof = std::max(h->max_ndof, P.body[i].ndof);
         h->has_3dof = h->has_3dof || P.body[i].sub != MB_SUB_SIX;
      }
      for (int i = 0; i < P.nb; i++) h->max_children = std::max(h->max_children, nchild[i]);
      cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
      h->warp_ok = mb::warp_variant_supports(P);
      if (h->warp_ok)
      {
         if ((e = cudaMalloc(&h->d_prog, 3 * sizeof(MbProgram))) != cudaSuccess) return bail(e, "cudaMalloc(programs)");
         if ((e = cudaMemcpy(h->d_prog, h->tree.prog, 3 * sizeof(MbProgram), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "cudaMemcpy(programs)");
      }
      // crossover batch sizes: linear in the body count through the measured crossovers of A7 (7 bodies,
      // profiles/r01h_batch_sweep_graph.jsonl) and H37 (32 bodies, profiles/r01y_batch_sweep.jsonl: the thread-per-state walk
      // of one state now takes 49 / 96 / 98 us, the warp kernels cross it at 4.8 k / 3.9 k / 3.4 k states).
      // MECANO_B200_WARP_BELOW overrides all three
      h->warp_below[MB_RNEA] = 2048 + 80 * P.nb; h->warp_below[MB_ABA] = 1536 + 64 * P.nb; h->warp_below[MB_CRBA] = 2048 + 40 * P.nb;
      if (P.nb > 32)
      {
         // team-per-state kernels (team_kernels.cu), trees of 51 / 75 / 101 bodies: crossovers at 2.5-2.7 k (RNEA), 1.5-2.0 k (ABA)
         // and 3.3-4.5 k states (CRBA), profiles/r05b_config5_1gpu.jsonl
         h->warp_below[MB_RNEA] = 2560; h->warp_below[MB_ABA] = 1792; h->warp_below[MB_CRBA] = 3584;
      }
      if (const char *e = getenv("MECANO_B200_WARP_BELOW"))
         h->warp_below[0] = h->warp_below[1] = h->warp_below[2] = atoll(e);
   }
   *out = h;
   return MECANO_B200_OK;
}

void mecano_b200_destroy(mecano_b200_handle *h)
{
   if (!h) return;
   DeviceGuard device_guard_(h->device);
   for (int i = 0; i < MB_MAX_SLOTS; i++)
   {
      if (h->stage[i]) cudaFree(h->stage[i]);
      if (h->done[i]) cudaEventDestroy(h->done[i]);
      if (h->streams[i]) cudaStreamDestroy(h->streams[i]);
   }
   if (h->d_zero_row) cudaFree(h->d_zero_row);
   if (h->d_scratch) cudaFree(h->d_scratch);
   if (h->d_consts) cudaFree(h->d_consts);
   if (h->d_counters) cudaFree(h->d_counters);
   if (h->d_zero) cudaFree(h->d_zero);
   if (h->d_yzero) cudaFree(h->d_yzero);
   if (h->d_prog) cudaFree(h->d_prog);
   for (int i = 0; i < 1 + MB_MAX_SLOTS; i++)
      if (h->d_ws[i]) cudaFree(h->d_ws[i]);
   for (int i = 0; i < 3; i++)
      mb::spec_unload(h->spec[i]);
   delete h;
}

const char *mecano_b200_last_error(const mecano_b200_handle *h)
{
   if (h) return h->error.c_str();
   return g_create_error.c_str();
}

int mecano_b200_set_gravity(mecano_b200_handle *h, double gx, double gy, double gz)
{
   if (!h) return MECANO_B200_ERR_INVALID_ARGUMENT;
   h->gravity[0] = gx; h->gravity[1] = gy; h->gravity[2] = gz;
   return MECANO_B200_OK;
}

int mecano_b200_set_precision(mecano_b200_handle *h, int precision)
{
   if (!h || (precision != MECANO_B200_PRECISION_FP64 && precision != MECANO_B200_PRECISION_FP32)) return MECANO_B200_ERR_INVALID_ARGUMENT;
   h->fp32 = precision == MECANO_B200_PRECISION_FP32;
   return MECANO_B200_OK;
}

int mecano_b200_set_grid_limit(mecano_b200_handle *h, int algo, int max_blocks)
{
   if (!h || algo < 0 || algo >= MB_NUM_ALGOS || max_blocks < 0) return MECANO_B200_ERR_INVALID_ARGUMENT;
   h->grid_limit[algo] = max_blocks;
   return MECANO_B200_OK;
}

int mecano_b200_set_variant(mecano_b200_handle *h, int variant)
{
   if (!h) return MECANO_B200_ERR_INVALID_ARGUMENT;
   if (variant != MECANO_B200_VARIANT_AUTO && variant != MECANO_B200_VARIANT_THREAD && variant != MECANO_B200_VARIANT_WARP)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "unknown variant");
   if (variant == MECANO_B200_VARIANT_WARP && !h->warp_ok)
      return fail(h, MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY, "the warp-per-state variant (one lane per body) handles trees of one-DoF and SixDoF joints");
   h->variant = variant;
   return MECANO_B200_OK;
}

int mecano_b200_specialize(mecano_b200_handle *h, uint32_t algo_mask)
{
   if (!h) return MECANO_B200_ERR_INVALID_ARGUMENT;
   std::lock_guard<std::mutex> lk(h->mu);
   MB_ON_DEVICE(h);
   for (int algo = 0; algo < 3; algo++)
   {
      if (!(algo_mask & (1u << algo)) || h->spec[algo].ready())
         continue;
      if (algo == MB_CRBA)
         continue; // bound by the HBM write of the mass matrix (DESIGN.md): the generic kernel is already at the roof
      if (h->has_3dof)
         continue; // spherical / planar joints: the generic kernels serve them (two-slot pass-three records, multidof_aba.cuh)
      const MbProgram &P = h->tree.prog[algo];
      // Unrolled code is fetched once per tile of states; beyond ~100 KB it no longer fits the instruction caches and the
      // block becomes fetch-bound (measured: 32-body humanoid RNEA 172 KB -> 0.78x, 15-body tree 81 KB -> 1.42x of the generic
      // kernel; profiles/r01g_spec.jsonl).  Estimated size: RNEA ~5.4 KB, ABA ~12 KB of SASS per body.
      const double est_kb = h->tree.nb * (algo == MB_RNEA ? 5.4 : 12.0);
      if (est_kb > 110.0 && !(algo_mask & MECANO_B200_SPECIALIZE_FORCE))
         continue;
      mb::SpecOptions opt;
      // defaults from the launch-configuration sweep (profiles/): RNEA 16 warps with a TMEM stack, ABA 8 warps in shared memory
      if (algo == MB_RNEA) { opt.block = 512; opt.tm = 32; }
      else { opt.block = 256; opt.tm = 0; }
      spec_cfg_from_env(algo, opt);
      if (!mb_tm_fits(algo, P, opt.tm, opt.block))
         opt.tm = 0; // the wide stack area of a deep tree does not fit the TMEM columns of one warp: shared memory only
      if (opt.tm * 4 > (512 / ((opt.block + 127) / 128) & ~3))
         return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "MECANO_B200_SPEC_CFG: TMEM slots exceed the columns of one warp");
      std::string err;
      int rc = MECANO_B200_ERR_TOO_LARGE;
      // shrink the block until the shared-memory part of the stack fits
      for (int b = opt.block; b >= 64 && rc == MECANO_B200_ERR_TOO_LARGE; b >>= 1)
      {
         mb::SpecOptions o2 = opt;
         o2.block = b;
         o2.tm = opt.tm > 0 ? std::min(opt.tm * (opt.block / b), 128) : 0;
         if (!mb_tm_fits(algo, P, o2.tm, o2.block))
            o2.tm = 0;
         int max_optin = 0;
         cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device);
         if (mb::spec_smem_bytes(algo, P, o2.block, o2.tm) + 1024 > (size_t)max_optin)
            continue;
         rc = mb::spec_build(algo, h->tree, o2, h->spec[algo], err);
      }
      if (rc != MECANO_B200_OK)
         return fail(h, rc, "specialize: " + err);
   }
   return MECANO_B200_OK;
}

int mecano_b200_n_dofs(const mecano_b200_handle *h) { return h ? h->tree.nv : -1; }
int mecano_b200_n_cfg(const mecano_b200_handle *h) { return h ? h->tree.nq : -1; }
int mecano_b200_n_bodies(const mecano_b200_handle *h) { return h ? h->tree.nb : -1; }

int mecano_b200_rnea(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, const double *fext,
                     double *tau, uint32_t flags, void *stream)
{
   Job j;
   const int rc = rnea_job(h, n, ld, q, qd, qdd, fext, tau, nullptr, nullptr, flags, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_rnea_full(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, const double *fext,
                          double *tau, double *body_acc, double *joint_wrench, uint32_t flags, void *stream)
{
   Job j;
   const int rc = rnea_job(h, n, ld, q, qd, qdd, fext, tau, body_acc, joint_wrench, flags, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_aba(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau, const double *fext,
                    double *qdd, uint32_t flags, void *stream)
{
   Job j;
   const int rc = aba_job(h, n, ld, q, qd, tau, nullptr, fext, qdd, nullptr, flags, false, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_set_joint_source_modes(mecano_b200_handle *h, const int32_t *accel_source)
{
   if (!h) return MECANO_B200_ERR_INVALID_ARGUMENT;
   std::lock_guard<std::mutex> lk(h->mu);
   h->n_accel_source = mb::apply_source_modes(h->tree, accel_source, h->effort_dof_runs);
   return MECANO_B200_OK;
}

int mecano_b200_aba_sources(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau, const double *qdd_in,
                            const double *fext, double *qdd, double *tau_out, void *stream)
{
   Job j;
   const int rc = aba_job(h, n, ld, q, qd, tau, qdd_in, fext, qdd, tau_out, 0u, true, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_aba_sources_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau,
                                 const double *qdd_in, const double *fext, double *qdd, double *tau_out)
{
   // ahead of the shape checks, also on an empty batch (the device entry point refuses a missing qdd_in when it launches)
   if (h && h->n_accel_source > 0 && !qdd_in)
      return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer (qdd_in) with joints in ACCELERATION_SOURCE mode");
   Job j;
   const int rc = aba_job(h, n, ld, q, qd, tau, qdd_in, fext, qdd, tau_out, 0u, true, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_crba_centroidal(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, double *M, double *cmm, double *com, int frame,
                                void *stream)
{
   Job j;
   const int rc = centroidal_job(h, n, ld, q, M, cmm, com, frame, false, j);
   return rc ? rc : run_device(h, j, stream);
}

// The centre of mass alone (CenterOfMassCalculator.getCenterOfMass() / getTotalMass(), CenterOfMassCalculator.java:70-124; what
// CenterOfMassReferenceFrame.updateTransformToParent(), CenterOfMassReferenceFrame.java:45-50, asks for).
int mecano_b200_center_of_mass(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, double *com, void *stream)
{
   Job j;
   const int rc = centroidal_job(h, n, ld, q, nullptr, nullptr, com, MECANO_B200_FRAME_WORLD, true, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_centroidal_convective_term(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *com,
                                           double *out, int frame, void *stream)
{
   Job j;
   const int rc = convective_term_job(h, n, ld, q, qd, com, out, frame, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_coriolis(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, double *M, double *C, void *stream)
{
   Job j;
   const int rc = coriolis_job(h, n, ld, q, qd, M, C, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_coriolis_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, double *M, double *C)
{
   Job j;
   const int rc = coriolis_job(h, n, ld, q, qd, M, C, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_joint_torque_regressor(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, double *Y,
                                       void *stream)
{
   Job j;
   const int rc = regressor_job(h, n, ld, q, qd, qdd, Y, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_joint_torque_regressor_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, double *Y)
{
   Job j;
   const int rc = regressor_job(h, n, ld, q, qd, qdd, Y, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_gravity_gradient(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *fext, double *tau, double *G, void *stream)
{
   Job j;
   const int rc = gravity_gradient_job(h, n, ld, q, fext, tau, G, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_gravity_gradient_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *fext, double *tau, double *G)
{
   Job j;
   const int rc = gravity_gradient_job(h, n, ld, q, fext, tau, G, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_rnea_derivatives(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, const double *fext,
                                 double *tau, double *dq, double *dqd, void *stream)
{
   Job j;
   const int rc = rnea_derivatives_job(h, n, ld, q, qd, qdd, fext, tau, dq, dqd, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_rnea_derivatives_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd,
                                      const double *fext, double *tau, double *dq, double *dqd)
{
   Job j;
   const int rc = rnea_derivatives_job(h, n, ld, q, qd, qdd, fext, tau, dq, dqd, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_aba_derivatives(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau, const double *fext,
                                double *qdd, double *dq, double *dqd, double *minv, void *stream)
{
   Job j;
   const int rc = aba_derivatives_job(h, n, ld, q, qd, tau, fext, qdd, dq, dqd, minv, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_aba_derivatives_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau,
                                     const double *fext, double *qdd, double *dq, double *dqd, double *minv)
{
   Job j;
   const int rc = aba_derivatives_job(h, n, ld, q, qd, tau, fext, qdd, dq, dqd, minv, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_crba_centroidal_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, double *M, double *cmm, double *com, int frame)
{
   Job j;
   const int rc = centroidal_job(h, n, ld, q, M, cmm, com, frame, false, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_centroidal_convective_term_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *com,
                                                double *out, int frame)
{
   Job j;
   const int rc = convective_term_job(h, n, ld, q, qd, com, out, frame, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_center_of_mass_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, double *com)
{
   Job j;
   const int rc = centroidal_job(h, n, ld, q, nullptr, nullptr, com, MECANO_B200_FRAME_WORLD, true, j);
   return rc ? rc : run_host(h, j);
}

// Not step_job: a caller's own buffer keeps ZEROS_PRESENT in every layout, and the kernel refuses what the layout does not combine with.
int mecano_b200_crba(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, double *M, uint32_t layout, void *stream)
{
   int rc = check_batch(h, n, ld);
   if (rc) return rc;
   if (n == 0) return MECANO_B200_OK;
   if (!q || !M) return fail(h, MECANO_B200_ERR_INVALID_ARGUMENT, "NULL buffer");
   MB_ON_DEVICE(h);
   return run(h, MB_CRBA, n, ld, q, nullptr, nullptr, nullptr, M, layout, (cudaStream_t)stream);
}

int mecano_b200_rnea_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd,
                          const double *fext, double *tau, uint32_t flags)
{
   return mecano_b200_rnea_full_host(h, n, ld, q, qd, qdd, fext, tau, nullptr, nullptr, flags);
}

int mecano_b200_rnea_full_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd,
                               const double *fext, double *tau, double *body_acc, double *joint_wrench, uint32_t flags)
{
   Job j;
   const int rc = rnea_job(h, n, ld, q, qd, qdd, fext, tau, body_acc, joint_wrench, flags, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_aba_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau,
                         const double *fext, double *qdd, uint32_t flags)
{
   Job j;
   const int rc = aba_job(h, n, ld, q, qd, tau, nullptr, fext, qdd, nullptr, flags, false, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_integrate(mecano_b200_handle *h, int64_t n, int64_t ld, double dt, double *q, double *qd, double *qdd, void *stream)
{
   Job j;
   const int rc = integrate_job(h, n, ld, dt, q, qd, qdd, j);
   return rc ? rc : run_device(h, j, stream);
}

int mecano_b200_integrate_host(mecano_b200_handle *h, int64_t n, int64_t ld, double dt, double *q, double *qd, double *qdd)
{
   Job j;
   const int rc = integrate_job(h, n, ld, dt, q, qd, qdd, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_crba_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, double *M, uint32_t layout)
{
   return mecano_b200_step_host(h, n, ld, q, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, M, layout);
}

int mecano_b200_crba_packed_size(const mecano_b200_handle *h) { return h ? (int)h->tree.packed_row.size() : -1; }

int mecano_b200_crba_packed_index(const mecano_b200_handle *h, int32_t *row, int32_t *col)
{
   if (!h) return MECANO_B200_ERR_INVALID_ARGUMENT;
   if (row) std::copy(h->tree.packed_row.begin(), h->tree.packed_row.end(), row);
   if (col) std::copy(h->tree.packed_col.begin(), h->tree.packed_col.end(), col);
   return MECANO_B200_OK;
}

int mecano_b200_step_host(mecano_b200_handle *h, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd_in, const double *tau_in,
                          const double *fext, double *tau_out, double *qdd_out, double *M, uint32_t layout)
{
   Job j;
   const int rc = step_job(h, n, ld, q, qd, qdd_in, tau_in, fext, tau_out, qdd_out, M, layout, j);
   return rc ? rc : run_host(h, j);
}

int mecano_b200_kernel_info_get(mecano_b200_handle *h, int algo, int64_t n_states, mecano_b200_kernel_info *info)
{
   if (!h || !info || algo < 0 || algo >= MB_NUM_ALGOS) return MECANO_B200_ERR_INVALID_ARGUMENT;
   const bool warp = !mb_algo(algo).thread_only && (h->variant == MECANO_B200_VARIANT_WARP || (h->variant == MECANO_B200_VARIANT_AUTO && h->warp_ok && n_states > 0 && n_states < h->warp_below[algo]));
   if (warp)
   {
      std::memset(info, 0, sizeof *info);
      cudaFuncAttributes fa;
      const bool team = h->tree.prog[algo].nb > 32;
      if (team) MB_CUDA(h, mb::team_kernel_attributes(algo, false, &fa));
      else MB_CUDA(h, mb::warp_kernel_attributes(algo, false, &fa));
      info->variant = MECANO_B200_VARIANT_WARP;
      info->block_threads = team ? mb::team_threads(h->tree.prog[algo]) : 128;
      info->states_per_block = team ? 1 : 4;
      info->regs_per_thread = fa.numRegs;
      info->local_bytes_per_thread = (int32_t)fa.localSizeBytes;
      info->static_smem_bytes = (int32_t)fa.sharedSizeBytes;
      info->sm_count = h->sm_count;
      info->max_depth = h->tree.prog[algo].max_depth;
      info->bytes_per_state = bytes_per_state(algo, h->tree.nq, h->tree.nv, h->tree.prog[algo].nb);
      return MECANO_B200_OK;
   }
   const mb::LaunchPlan &p = h->plan[algo];
   const MbProgram &P = h->tree.prog[algo];
   std::memset(info, 0, sizeof *info);
   info->variant = MECANO_B200_VARIANT_THREAD;
   const mb::SpecKernel &sk = h->spec[algo];
   if (sk.ready())
   {
      info->block_threads = sk.opt.block;
      info->states_per_block = sk.opt.block;
      info->regs_per_thread = sk.regs;
      info->static_smem_bytes = sk.static_smem;
      info->dynamic_smem_bytes = (int32_t)sk.smem;
      info->local_bytes_per_thread = sk.local_bytes;
      info->blocks_per_sm = sk.blocks_per_sm;
      info->specialized = 1 + (sk.from_cache ? 1 : 0);
      info->tmem_stack_slots = sk.opt.tm;
      info->jit_seconds = sk.compile_seconds;
   }
   else
   {
      info->block_threads = p.block;
      info->states_per_block = p.block;
      info->regs_per_thread = p.regs;
      info->static_smem_bytes = p.static_smem;
      info->dynamic_smem_bytes = (int32_t)p.smem;
      info->local_bytes_per_thread = p.local_bytes;
      info->blocks_per_sm = p.blocks_per_sm;
      info->tmem_stack_slots = p.tm;
   }
   cudaDeviceGetAttribute(&info->sm_count, cudaDevAttrMultiProcessorCount, h->device);
   info->stack_doubles = P.stack_doubles;
   info->max_depth = P.max_depth;
   info->bytes_per_state = bytes_per_state(algo, P.nq, P.nv, P.nb);
   return MECANO_B200_OK;
}

int mecano_b200_measure_fp64_peak(int device, double *tflops)
{
   if (!tflops) return MECANO_B200_ERR_INVALID_ARGUMENT;
   cudaError_t e = cudaSetDevice(device);
   if (e == cudaSuccess) e = mb::measure_fp64_peak(tflops);
   return e == cudaSuccess ? MECANO_B200_OK : (int)e;
}

int mecano_b200_measure_fp64_sustained(int device, double seconds, double *tflops)
{
   if (!tflops || !(seconds > 0.0) || seconds > 30.0) return MECANO_B200_ERR_INVALID_ARGUMENT;
   cudaError_t e = cudaSetDevice(device);
   if (e == cudaSuccess) e = mb::measure_fp64_sustained(seconds, tflops);
   return e == cudaSuccess ? MECANO_B200_OK : (int)e;
}

int mecano_b200_measure_hbm_peak(int device, double *gbs)
{
   if (!gbs) return MECANO_B200_ERR_INVALID_ARGUMENT;
   cudaError_t e = cudaSetDevice(device);
   if (e == cudaSuccess) e = mb::measure_hbm_peak(gbs);
   return e == cudaSuccess ? MECANO_B200_OK : (int)e;
}

int mecano_b200_generate_source(const mecano_b200_tree_desc *desc, int algo, int block_threads, int tmem_slots, char *buf, int64_t capacity, int64_t *needed)
{
   if (algo < 0 || algo > 2) return fail(nullptr, MECANO_B200_ERR_INVALID_ARGUMENT, "algo must be 0 (RNEA), 1 (ABA) or 2 (CRBA)");
   mb::FlatTree tree;
   std::string err;
   int rc = mb::flatten_tree(desc, tree, err);
   if (rc != MECANO_B200_OK) return fail(nullptr, rc, err);
   mb::SpecOptions opt;
   opt.block = block_threads > 0 ? block_threads : 256;
   opt.tm = tmem_slots;
   const std::string src = mb::generate_source(algo, tree, opt);
   if (needed) *needed = (int64_t)src.size() + 1;
   if (buf && capacity > 0)
   {
      const size_t n = std::min<size_t>(src.size(), (size_t)capacity - 1);
      std::memcpy(buf, src.data(), n);
      buf[n] = 0;
   }
   return MECANO_B200_OK;
}

int mecano_b200_jit_check(const mecano_b200_tree_desc *desc, int algo, int block_threads, int tmem_slots, int64_t *cubin_bytes)
{
   if (algo < 0 || algo > 2) return fail(nullptr, MECANO_B200_ERR_INVALID_ARGUMENT, "algo must be 0 (RNEA), 1 (ABA) or 2 (CRBA)");
   mb::FlatTree tree;
   std::string err;
   int rc = mb::flatten_tree(desc, tree, err);
   if (rc != MECANO_B200_OK) return fail(nullptr, rc, err);
   mb::SpecOptions opt;
   opt.block = block_threads > 0 ? block_threads : 256;
   opt.tm = tmem_slots;
   size_t bytes = 0;
   rc = mb::spec_compile_only(mb::generate_source(algo, tree, opt), &bytes, err);
   if (cubin_bytes) *cubin_bytes = (int64_t)bytes;
   if (rc != MECANO_B200_OK) return fail(nullptr, rc, err);
   return MECANO_B200_OK;
}

int mecano_b200_host_alloc(void **ptr, int64_t bytes)
{
   if (!ptr || bytes < 0) return MECANO_B200_ERR_INVALID_ARGUMENT;
   cudaError_t e = cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocDefault);
   return e == cudaSuccess ? MECANO_B200_OK : (int)e;
}

int mecano_b200_host_free(void *ptr)
{
   cudaError_t e = cudaFreeHost(ptr);
   return e == cudaSuccess ? MECANO_B200_OK : (int)e;
}

// ------------------------------------------------------------------------------------------------ several devices, one call
#pragma GCC visibility pop
} // extern "C"

struct mecano_b200_multi
{
   std::vector<mecano_b200_handle *> lanes;
   std::string error;
};

namespace
{
// slice of lane i: contiguous, multiples of 256 states (aligned rows on the device side), the remainder on the last lanes
void multi_slice(int64_t n, int lanes, int i, int64_t *start, int64_t *count)
{
   const int64_t blocks = (n + 255) / 256, base = blocks / lanes, extra = blocks % lanes;
   const int64_t b0 = (int64_t)i * base + std::min<int64_t>(i, extra), b1 = b0 + base + (i < extra ? 1 : 0);
   *start = std::min(n, b0 * 256);
   *count = std::min(n, b1 * 256) - *start;
}

int multi_fail(mecano_b200_multi *m, int rc, int lane)
{
   if (rc && m && lane >= 0 && lane < (int)m->lanes.size())
      m->error = "device entry " + std::to_string(lane) + " (cuda:" + std::to_string(m->lanes[(size_t)lane]->device) + "): " + m->lanes[(size_t)lane]->error;
   return rc;
}

// One job per lane from the whole-batch job that `build` checks and declares on the first lane's handle: every pointer offset to the
// lane's first state (state-major outputs by whole states).
template <class Build>
int multi_run(mecano_b200_multi *m, int64_t n, int64_t ld, const Build &build)
{
   if (!m) return MECANO_B200_ERR_INVALID_ARGUMENT;
   if (n < 0 || ld < n)
   {
      m->error = "n_states must be >= 0 and ld >= n_states";
      return MECANO_B200_ERR_SHAPE;
   }
   Job whole;
   int rc = build(m->lanes[0], whole);
   if (rc) return multi_fail(m, rc, 0);
   const int L = (int)m->lanes.size();
   std::vector<Job> jobs((size_t)L, whole);
   for (int i = 0; i < L; i++)
   {
      int64_t s0 = 0, cnt = 0;
      multi_slice(n, L, i, &s0, &cnt);
      Job &j = jobs[(size_t)i];
      j.n = cnt;
      j.variant_n = n;
      for (JobIn &in : j.in)
         if (in.host) in.host += s0;
      for (JobStep &st : j.steps)
         for (JobOut &o : st.out)
            if (o.host) o.host += o.how == COPY_STATES ? (size_t)s0 * o.rows : (size_t)s0;
   }
   int failed = 0;
   rc = run_host_lanes(m->lanes, jobs, &failed);
   return multi_fail(m, rc, failed);
}
} // namespace

extern "C" {
#pragma GCC visibility push(default)

int mecano_b200_multi_create(const mecano_b200_tree_desc *desc, const int32_t *devices, int n_devices, mecano_b200_multi **out)
{
   if (!out) return fail(nullptr, MECANO_B200_ERR_INVALID_ARGUMENT, "out pointer is NULL");
   *out = nullptr;
   if (!devices || n_devices <= 0 || n_devices > 64) return fail(nullptr, MECANO_B200_ERR_INVALID_ARGUMENT, "device list must hold 1 .. 64 entries");
   mecano_b200_multi *m = new mecano_b200_multi();
   for (int i = 0; i < n_devices; i++)
   {
      mecano_b200_handle *h = nullptr;
      const int rc = mecano_b200_create(desc, devices[i], &h);
      if (rc != MECANO_B200_OK)
      {
         mecano_b200_multi_destroy(m);
         return rc; // mecano_b200_last_error(NULL) holds the message of the failed create
      }
      m->lanes.push_back(h);
   }
   *out = m;
   return MECANO_B200_OK;
}

void mecano_b200_multi_destroy(mecano_b200_multi *m)
{
   if (!m) return;
   for (mecano_b200_handle *h : m->lanes) mecano_b200_destroy(h);
   delete m;
}

const char *mecano_b200_multi_last_error(const mecano_b200_multi *m) { return m ? m->error.c_str() : mecano_b200_last_error(nullptr); }
int mecano_b200_multi_size(const mecano_b200_multi *m) { return m ? (int)m->lanes.size() : -1; }
mecano_b200_handle *mecano_b200_multi_handle(mecano_b200_multi *m, int i) { return (m && i >= 0 && i < (int)m->lanes.size()) ? m->lanes[(size_t)i] : nullptr; }

int mecano_b200_multi_slice(const mecano_b200_multi *m, int64_t n_states, int i, int64_t *start, int64_t *count)
{
   if (!m || i < 0 || i >= (int)m->lanes.size() || n_states < 0 || !start || !count) return MECANO_B200_ERR_INVALID_ARGUMENT;
   multi_slice(n_states, (int)m->lanes.size(), i, start, count);
   return MECANO_B200_OK;
}

int mecano_b200_multi_set_gravity(mecano_b200_multi *m, double gx, double gy, double gz)
{
   if (!m) return MECANO_B200_ERR_INVALID_ARGUMENT;
   for (mecano_b200_handle *h : m->lanes) mecano_b200_set_gravity(h, gx, gy, gz);
   return MECANO_B200_OK;
}

int mecano_b200_multi_rnea_host(mecano_b200_multi *m, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd, const double *fext,
                                double *tau, uint32_t flags)
{
   return multi_run(m, n, ld, [&](mecano_b200_handle *h, Job &j) { return rnea_job(h, n, ld, q, qd, qdd, fext, tau, nullptr, nullptr, flags, j); });
}

int mecano_b200_multi_aba_host(mecano_b200_multi *m, int64_t n, int64_t ld, const double *q, const double *qd, const double *tau, const double *fext,
                               double *qdd, uint32_t flags)
{
   return multi_run(m, n, ld, [&](mecano_b200_handle *h, Job &j) { return aba_job(h, n, ld, q, qd, tau, nullptr, fext, qdd, nullptr, flags, false, j); });
}

int mecano_b200_multi_crba_host(mecano_b200_multi *m, int64_t n, int64_t ld, const double *q, double *M, uint32_t layout)
{
   return mecano_b200_multi_step_host(m, n, ld, q, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, M, layout);
}

int mecano_b200_multi_step_host(mecano_b200_multi *m, int64_t n, int64_t ld, const double *q, const double *qd, const double *qdd_in, const double *tau_in,
                                const double *fext, double *tau_out, double *qdd_out, double *M, uint32_t layout)
{
   return multi_run(m, n, ld, [&](mecano_b200_handle *h, Job &j) {
      return step_job(h, n, ld, q, qd, qdd_in, tau_in, fext, tau_out, qdd_out, M, layout, j);
   });
}

#pragma GCC visibility pop
} // extern "C"
