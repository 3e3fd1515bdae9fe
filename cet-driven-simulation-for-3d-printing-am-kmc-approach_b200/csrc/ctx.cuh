// ctx.cuh — the lattice context behind the opaque `cet_ctx` of include/cetkmc.h, and the
// error plumbing shared by all translation units.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <vector>
#include "../../include/cetkmc.h"
#include "site_rates.cuh"

namespace cet {

void set_error(const char *fmt, ...);

#define CET_CUDA(call)                                                                     \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            cet::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return 1000 + (int)e_;                                                         \
        }                                                                                  \
    } while (0)

#define CET_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            cet::set_error(__VA_ARGS__);  \
            return 1;                     \
        }                                 \
    } while (0)

// Counters that live in device memory and are advanced by the single-CTA step kernel.
struct KmcState {
    int64_t steps_done, py_pos, np_pos, sp_pos, nucleation_count, fallback_last;
    double total_time, last_total_rate;
    int32_t terminated, starved;
};

// One changed boundary-zone site of a sweep, as its owner sends it to the neighbouring slab.
struct DeltaEntry {
    double theta, phi;
    int32_t zidx;        // (plane within the 6-plane zone) * plane_sites + in-plane index
    uint32_t vox;        // the packed voxel byte
};
constexpr int DELTA_ZONE = 6;      // planes per face a neighbour keeps as ghosts (= SWEEP_HALO)
constexpr int DELTA_HEADER = 16;   // bytes in front of the entries; the first 4 hold the count

// Three 128-byte lines, by who touches them while a kernel runs: a read of a line that thousands of atomics
// are queued on waits behind them, and every CTA of the sweep kernels starts by reading tau or n_fired.
struct SweepState {
    // line 0 — running totals over owned sites, advanced by device atomics at the end of the apply CTAs
    unsigned long long n_fired_total, n_applied, n_nuc;
    unsigned long long n_refreshed_total;                 // sites re-evaluated by the neighbour-rate refresh
    unsigned long long pad_line0_[12];
    // line 1 — list reservations (atomics of the stream / scan kernels), read by the kernels that follow
    unsigned int n_fired;                           // fired-site list length of the current sweep
    unsigned int n_dirty, n_dirty_emp;              // refresh list length (one mixed list; n_dirty_emp stays 0, kept for the layout)
    unsigned int overflow, dirty_overflow, pad0_;   // the fired list overflowed (events dropped)
    unsigned int pad_line1_[26];
    // line 2 — written by the single-CTA finalize kernel only
    double sum_rate, max_rate;                      // totals of the rates seen by the last sweep
    double tau, time;                               // interval of the next sweep; accumulated time
    int32_t terminated, pad_;
    unsigned long long pad_line2_[11];
};
static_assert(offsetof(SweepState, n_fired) == 128 && offsetof(SweepState, sum_rate) == 256 && sizeof(SweepState) == 384,
              "SweepState: one 128-byte line per access class");

// Grouped sweeps (cet_sweep_run_group): one launch covers the lattices of a group, and a CTA takes the
// arguments of its lattice (blockIdx.z, or blockIdx.x for the one-CTA kernels) from a table passed by value
// in kernel parameter space (32 KB).  CAP is the table's capacity: a launch copies the whole table, so a
// small group uses the small one.
constexpr int GROUP_MAX = 64;
template <class T, int CAP>
struct GroupArgs {
    T a[CAP];
};
template <class T>
constexpr bool group_fits() { return sizeof(GroupArgs<T, GROUP_MAX>) <= 32764; }

}  // namespace cet

// Device-memory layout (all arrays cover local planes [0, np) where np = ni + 2*halo and local
// plane p holds global plane i_begin - halo + p; k is the fastest axis, then j, then plane):
//   vox        u8   np*n1*n2   state | defects<<4
//   vox_prev   u8   np*n1*n2   snapshot for the latent-heat term (allocated on first use)
//   theta,phi  f64  np*n1*n2
//   v          4xf64 np*n1*n2  orientation unit vectors, one 32-byte record per site (derived from theta/phi; kept in step by every
//                              writer of theta/phi so the rate kernels never call sin/cos)
//   T, T2      f64  np*n1*n2   ping-pong buffers of the thermal stencil
//   site_rate  f64  np*n1*n2   sum of the site's diff (occupied) or nuc+att (empty) rates
//   dep_rate   f64  n1*n2      top plane only: deposition rate, NaN where no dep event exists
//   row_occ / row_emp  f64  np*n1   per (plane, j) row sums split by occupancy class
//   row_dep    f64  n1 ; row_depcnt i32 n1
//   seg        f64  3*np       per-plane segment sums in list order: dep | occupied | empty
//   total      f64  1 (+ n_dep i64)
struct cet_ctx {
    int device = 0;
    int64_t n0 = 0, n1 = 0, n2 = 0;   // global extents (rates require n0 == n1 == n2 == L)
    int64_t i_begin = 0, i_end = 0;   // owned global planes
    int halo = 0;
    int64_t np = 0;                   // local planes incl. ghosts
    int64_t plane = 0;                // n1*n2
    int64_t nloc = 0;                 // np*plane
    bool cubic = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;

    uint8_t *vox = nullptr, *vox_prev = nullptr;
    double *theta = nullptr, *phi = nullptr, *T = nullptr, *T2 = nullptr;
    cet::Vec4 *v = nullptr;
    uint64_t *nst = nullptr;          // neighbour-state cache (see site_rates.cuh); valid on planes with both i-neighbour pairs local
    bool nst_valid = false;
    double *site_rate = nullptr, *dep_rate = nullptr;
    double *row_occ = nullptr, *row_emp = nullptr, *row_dep = nullptr, *seg = nullptr;
    int32_t *row_depcnt = nullptr;
    double *total = nullptr;          // [0] total, [1] (as int64) n_dep
    double *q_top = nullptr;
    bool T_finite = false;            // T holds no NaN/inf (set by a nan_to_num stencil pass, cleared by uploads)
    bool rates_valid = false;         // site_rate / dep_rate and the BKL sum hierarchy valid on the owned planes
    bool sweep_rates_valid = false;   // site_rate / dep_rate valid on the planes the sweep evaluates

    // staging for host<->device conversion (grown on demand)
    void *stage = nullptr;
    size_t stage_bytes = 0;

    cet_rate_params rp{};
    bool have_rp = false;
    double *rate_tab = nullptr;       // K_eff / E_tot tables of rate_tile.cuh
    bool rate_tab_valid = false, rate_attr_set = false;

    // exact KMC
    cet::KmcState *kmc = nullptr;
    double *d_py = nullptr, *d_np = nullptr, *d_sp = nullptr;
    size_t cap_py = 0, cap_np = 0, cap_sp = 0;
    void *d_log = nullptr;
    size_t cap_log = 0;

    // sweep mode
    uint32_t *stamp = nullptr;        // refresh requests of the current sweep, one bit per local site
    int32_t *dirty = nullptr, *fired = nullptr;
    size_t cap_dirty = 0, cap_fired = 0;
    cet::SweepState *sweep = nullptr;
    unsigned long long *claim = nullptr;
    void *records = nullptr;
    size_t cap_records = 0;
    int64_t sweep_index = 0;
    int64_t last_thermal_index = -1;  // sweep index whose thermal step has already run (priming pass)
    double *blk_sum = nullptr, *blk_max = nullptr, *plane_sum = nullptr;
    int64_t n_blk = 0;

    // fused tile kernel (sweep_tile.cu): resident class codes + pair operands, TMA descriptors
    uint8_t *cvox = nullptr;
    double *pairop = nullptr;
    int *tile_flag = nullptr;
    bool tile_valid = false;          // cvox / pairop match vox / theta / phi / T / defects / the state ids
    bool emp_canonical = false;       // no empty site carries an orientation (checked by tile_state_ensure)
    int tile_blocks[6] = {0, 0, 0, 0, 0, 0};   // resident CTAs per SM of the rates_tile3d_kernel variants (0 = not yet queried)
    int refresh_blocks[3] = {0, 0, 0};   // resident CTAs per SM of rates_refresh_kernel<1 / 2 / 4> (0 = not yet queried)
    int dense_blocks[2] = {0, 0};     // resident CTAs per SM of rates_dense_kernel<unsorted>, <sorted> (0 = not yet queried)
    bool compact_attr_set = false;    // shared-memory attribute of the pair-compacting kernels set
    int debug_flags = 0;              // cet_debug_flags: kernel variants for tests / profiling, bit values in include/cetkmc.h
    alignas(64) unsigned char tmap_vox[128];
    alignas(64) unsigned char tmap_po[128];
    const void *tmap_vox_ptr = nullptr, *tmap_po_ptr = nullptr;
    int n_sm = 0;                     // multiprocessors of the device (queried once)

    // grain clustering (grains.cu)
    int *grain_label = nullptr, *grain_gid = nullptr;
    int64_t n_grains = 0;
    int grain_p_lo = 0, grain_p_hi = 0;   // local planes the last labelling covered
    // grouped metrics cadence (metrics_group.cu), grow-only
    void *grain_st = nullptr;         // per-grain statistics in site order of the roots + pairwise leaf sums of the aspect ratios
    size_t cap_grain_st = 0;
    void *group_tab = nullptr;        // result table of the groups this context leads (GROUP_MAX entries)
    cudaEvent_t ev_group = nullptr;   // orders this context's stream before the work of a group led by another context
    void *profile_tab = nullptr;      // grain-profile tables and span differences of the groups this context leads, grow-only
    size_t cap_profile_tab = 0;

    // per-kernel-kind device timing (cet_profile_*): event pairs recorded around the dominant
    // kernels on the context stream, resolved when the totals are read
    bool profile = false;
    std::vector<cudaEvent_t> prof_pool;
    struct ProfSpan { int kind; cudaEvent_t a, b; };
    std::vector<ProfSpan> prof_spans;

    // NCCL
    void *nccl_comm = nullptr;
    void *nccl_comm2 = nullptr;       // split-off communicator for the totals reduction of the sweeps, on stream2 (NULL: none)
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_reduce_ready = nullptr, ev_reduce_done = nullptr;
    int rank = 0, world = 1;
    // delta halo exchange of the sweeps (comm.cu): per cut face one send and one receive buffer,
    // [0] lower face, [1] upper face; layout: 16-byte header (entry count) + DeltaEntry[delta_cap]
    void *delta_send[2] = {nullptr, nullptr}, *delta_recv[2] = {nullptr, nullptr};
    int64_t delta_cap = 0;

    cet::Lat lat() const
    {
        cet::Lat g;
        g.vox = vox; g.nst = nst; g.v = v; g.T = T;
        g.L = (int)n1; g.n0 = (int)n0;
        g.i_off = (int)(i_begin - halo);
        return g;
    }
    int64_t owned_offset() const { return (int64_t)halo * plane; }
    int64_t owned_sites() const { return (i_end - i_begin) * plane; }
};

namespace cet {
int ensure_stage(cet_ctx *c, size_t bytes);
int orient_update(cet_ctx *c, int64_t p_lo, int64_t p_hi);
int nst_build(cet_ctx *c, int p_lo, int p_hi);     // rebuild the neighbour-state cache of local planes [p_lo, p_hi)
int nst_ensure(cet_ctx *c);                          // ... of every plane it can be built for, if it is stale
int sm_count(cet_ctx *c);                            // multiprocessors of the context's device
// groups of contexts (metrics_group.cu): the common argument checks (distinct whole-lattice cubic contexts of one L
// on one device, 1 <= n_ctx <= GROUP_MAX), and the order of the group's work on ctxs[0]'s stream after the work
// already queued on every member's stream
int group_check(const char *fn, cet_ctx *const *ctxs, int32_t n_ctx);
int group_order(cet_ctx *const *ctxs, int n);
// every writer of vox / theta / phi / T / defects other than the tile-aware sweep kernels calls this
inline void lattice_changed(cet_ctx *c) { c->tile_valid = false; c->rates_valid = false; c->sweep_rates_valid = false; }
enum { PROF_DECIDE = 0, PROF_APPLY = 1, PROF_THERMAL = 2, PROF_RATES = 3, PROF_HALO = 4, PROF_STEP = 5, PROF_PICK = 6,
       PROF_REFRESH = 7, PROF_ALLREDUCE = 8, PROF_BOUNDARY = 9, PROF_KINDS = 10 };
// RAII span: records an event pair around a launch when profiling is on.
struct ProfScope {
    cet_ctx *c; int kind; cudaEvent_t a = nullptr;
    ProfScope(cet_ctx *ctx, int k) : c(ctx), kind(k)
    {
        if (!c->profile) return;
        if (c->prof_pool.empty()) { if (cudaEventCreate(&a) != cudaSuccess) { a = nullptr; return; } }
        else { a = c->prof_pool.back(); c->prof_pool.pop_back(); }
        cudaEventRecord(a, c->stream);
    }
    ~ProfScope()
    {
        if (!a) return;
        cudaEvent_t b = nullptr;
        if (c->prof_pool.empty()) { if (cudaEventCreate(&b) != cudaSuccess) { c->prof_pool.push_back(a); return; } }
        else { b = c->prof_pool.back(); c->prof_pool.pop_back(); }
        cudaEventRecord(b, c->stream);
        c->prof_spans.push_back({kind, a, b});
    }
};
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard()
    {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};
}  // namespace cet
