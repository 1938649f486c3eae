// skb_matvec.cu -- device-resident flow() layer (include/skelly_b200_flow.h): FiberContainer / Periphery /
// BodyContainer flows of SkellySim and their fused sum, the hydrodynamic part of System::apply_matvec
// (src/core/system.cpp:284-316).  Built on the pair-kernel contexts of skb_runtime.cu; everything between the
// upload of the strengths and the download of the velocities stays on the device.
#include "aux_kernels.cuh"
#include "fiber_ops.cuh"
#include "group_kernels.cuh"
#include "skb_internal.hpp"
#include "../../include/skelly_b200_flow.h"
#include "../../include/skelly_b200_dense.h"

#include <cmath>
#include <condition_variable>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace skb;

#define CUDA_TRY(expr)                                                                                                \
    do {                                                                                                              \
        cudaError_t _e = (expr);                                                                                      \
        if (_e != cudaSuccess)                                                                                        \
            return set_error(SKB_ERR_CUDA, "%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,                      \
                             cudaGetErrorString(_e));                                                                 \
    } while (0)
#define SKB_TRY(expr)                                                                                                 \
    do {                                                                                                              \
        int _rc = (expr);                                                                                             \
        if (_rc != SKB_OK)                                                                                            \
            return _rc;                                                                                               \
    } while (0)

namespace {
// reference defaults of the regularised helpers (include/kernels.hpp:38-46): reg = 5e-3, eps = 1e-5
constexpr double kReg = 5e-3;
constexpr double kEps = 1e-5;

struct TargetCache {
    std::vector<double> host;
    bool valid = false;
    unsigned long long version = 0; // bumped by every upload: part of the CUDA-graph key (a replay bakes in whether
                                    // the symmetric path -- targets start with the sources -- was taken)
    bool same(const double *r, long long n) const {
        return valid && (long long)host.size() == 3 * n && (n == 0 || std::memcmp(host.data(), r, (size_t)n * 24) == 0);
    }
    void store(const double *r, long long n) {
        host.assign(r, r + 3 * n);
        valid = true;
        ++version;
    }
};
} // namespace

struct skb_flow {
    int dev = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evt0 = nullptr, evt1 = nullptr;
    // geometry
    long long n_fib = 0, n_shell = 0, n_body = 0;
    int n_fibers = 0, n_bodies = 0, max_fiber_nodes = 0;
    DevBuf fiber_offset, fiber_length, r_fib, r_shell, r_body, centers;
    std::vector<double> h_r_fib, h_r_shell, h_r_body; // host copies to assemble the matvec target lists
    // evaluators: [0] arbitrary targets, [1] matvec target lists
    skb_ctx *fib[2] = {nullptr, nullptr}, *shell[2] = {nullptr, nullptr}, *body[2] = {nullptr, nullptr};
    TargetCache tc_fib, tc_shell, tc_body;
    bool mv_dirty = true;
    int cross_mode = -1;    // fiber <-> periphery cross kernel in the matvec: -1 auto, 0 off, 1 on whenever applicable
    bool use_cross = false; // decided by prepare_matvec_targets
    CrossState cross;
    bool self_excl = false; // matvec: skip intra-fiber pairs in the kernels instead of compute-then-subtract (N3, opt-in)
    long long win_begin = 0, win_end = -1; // target window of the matvec in [fibers|shell|bodies] rows; -1 = all
    bool use_ranges = false;               // skb_flow_set_target_ranges instead of a contiguous window
    long long rq_f0 = 0, rq_f1 = 0, rq_s0 = 0, rq_s1 = 0, rq_b0 = 0, rq_b1 = 0; // requested (fiber indices, rows)
    // resolved pieces of the matvec target list: fiber rows [fa,fb), shell rows [sa,sb), body rows [ba,bb);
    // the output has n_win = (fb-fa)+(sb-sa)+(bb-ba) rows in that order
    long long fa = 0, fb = 0, sa = 0, sb = 0, ba = 0, bb = 0, n_win = 0;
    int op_f0 = 0, op_f1 = 0; // fibers [op_f0, op_f1) whose operators are resident (the fiber rows of the target list)
    cudaStream_t cur = nullptr;            // stream of the call in flight (own stream or the caller's)
    int n_points = 0;
    DevBuf pt_pos, pt_force, pt_torque;
    bool has_background = false;
    // CUDA-graph replay of the launch-bound small-size calls (BASELINE C1, listener / streamline path)
    struct GraphSlot {
        cudaGraphExec_t exec = nullptr;
        unsigned long long key = 0, seen = 0;
        int launches = 0;
        long long pairs = 0;
        void reset() {
            if (exec)
                cudaGraphExecDestroy(exec);
            exec = nullptr;
            key = seen = 0;
        }
    } g_matvec, g_vat;
    unsigned long long geom_version = 1;
    bool graphs_enabled = true;
    double *h_stage = nullptr; // pinned staging: the graph's memcpy nodes need fixed host addresses
    size_t h_stage_cap = 0;
    int bg_comp[3] = {0, 1, 2};
    double bg_scale[3] = {0, 0, 0}, bg_uniform[3] = {0, 0, 0};
    // per-fiber dense operators (SURVEY.md §8f N2): A_, force_operator_, xs_ resident for the timestep
    std::vector<int> h_fiber_n;
    std::vector<long long> h_fiber_off;
    struct FiberClass {
        std::vector<double> D, P; // D_1_0 (n x n), P_downsample_bc ((4n-14) x 4n), column-major
    };
    std::map<int, FiberClass> fiber_classes;
    bool ops_ready = false;
    int n_items_A = 0, n_items_F = 0;
    size_t gemv_smem = 0;
    DevBuf op_A, op_F, op_xs, op_len, op_plus, op_class, op_classD, op_classP, op_classR, op_ranges, items_A, items_F;
    DevBuf x_fib, res_fib, vb, res_shell, op_Ainv, tmp_b;
    long long op_A_elems = 0;               // elements of the concatenated A_ (and of A_^-1)
    unsigned long long ops_gen = 0, precond_gen = 0; // the preconditioner belongs to one set of operators
    // multi-GPU group (group_kernels.cuh): one member per GPU, exchange through peer memory
    struct Group {
        int rank = 0, size = 1;
        void *window = nullptr;       // this member's window (cudaMalloc: exportable through CUDA IPC)
        size_t window_bytes = 0;
        void *peer[kMaxGroup] = {};   // base address of every member's window as mapped here (peer[rank] == window)
        bool peer_ipc[kMaxGroup] = {};
        size_t off_flags = 0, off_fsl[2] = {0, 0}, off_fshell[2] = {0, 0}, off_xshell[2] = {0, 0}, off_upart = 0;
        size_t off_upart_shell = 0;   // partial periphery velocities (cross kernel: own fibers -> ALL periphery rows)
        long long n_fib = 0, n_shell = 0, n_pad_fib = 0, n_pad_shell = 0; // geometry the window was laid out for
        unsigned long long epoch = 0;
        bool dry = false;             // warm-up pass: no flags, own window only (skb_flow_group_warmup)
        bool use_sym = false;         // fiber rows: symmetric block rows + pull-reduce (else own rows with the plain kernel)
        bool connected() const {
            for (int m = 0; m < size; ++m)
                if (!peer[m])
                    return false;
            return true;
        }
        template <class T> T *at(int member, size_t off) const { return reinterpret_cast<T *>((char *)peer[member] + off); }
    } grp;
    // Periphery::matvec's dense operator beside the pair kernels (stream_kernels.cuh): forked onto bg_stream once its
    // input (the complete x_shell) is there, joined before res_shell is assembled
    struct Overlap {
        bool enabled = true;       // skb_flow_set_overlap
        cudaStream_t stream = nullptr;
        cudaEvent_t fork = nullptr, join = nullptr;
        DevBuf y;                  // A x of the own periphery rows
        skb_dense *dn = nullptr;   // pending background product of the call in flight (nullptr: none)
        const double *d_x = nullptr;
        bool launched = false;
    } bg;
    DevBuf scratch_u; // group mode: landing zone of eval_on_device's default output (never read)
    // staging
    DevBuf in_fib, in_shell, in_body, in_force, in_torque, vel, tmp;
    skb_flow_stats stats{};
    int launches = 0;
    long long pairs = 0;
};

static int ensure_ctx(skb_flow *fl, skb_ctx **slot) {
    if (*slot)
        return SKB_OK;
    return skb_ctx_create_on(&fl->dev, 1, slot);
}

// bookkeeping of the n kernel launches just issued on behalf of fl
static int launched(skb_flow *fl, int n) {
    CUDA_TRY(cudaGetLastError());
    count_launch(n);
    fl->launches += n;
    return SKB_OK;
}

// ---- device-side flows: ctx already has its targets and sources ------------------------------------------------
// Self term of the fibers (fcfd.cpp:203-210) with Stokeslet strengths d_h: targets [0, node_end - node_begin) of d_v
// are the fiber nodes [node_begin, node_end).  Nothing to do in the opt-in fused form, where the pair kernels already
// skipped every intra-fiber pair (skb_flow_set_self_exclusion).
static int fiber_self_term(skb_flow *fl, const DeviceState &d, const double *d_h, double eta, double *d_v,
                           long long node_begin, long long node_end) {
    if (d.src[SKB_STOKESLET].excl)
        return SKB_OK;
    const size_t smem = (size_t)fl->max_fiber_nodes * 6 * sizeof(double);
    fiber_self_subtract_kernel<<<fl->n_fibers, 128, smem, fl->cur>>>(
        (const double *)fl->r_fib.ptr, d_h, (const long long *)fl->fiber_offset.ptr, 1.0 / (8.0 * M_PI * eta),
        kReg * kReg, kEps, d_v, node_begin, node_end);
    return launched(fl, 1);
}

// subtract_self: the first (node_end - node_begin) targets are the fiber nodes [node_begin, node_end)
static int fibers_dev(skb_flow *fl, skb_ctx *ctx, const double *d_forces, double eta, int subtract_self,
                      double *d_vel, int accumulate, long long node_begin, long long node_end) {
    DeviceState &d = ctx->devs[0];
    if (d.n_trg == 0)
        return SKB_OK;
    if (fl->n_fibers == 0) { // fiber_container_finite_difference.cpp:178-179
        if (!accumulate)
            CUDA_TRY(cudaMemsetAsync(d_vel, 0, (size_t)d.n_trg * 24, fl->cur));
        return SKB_OK;
    }
    // weighted forces -> Stokeslet all-to-all, / eta  (fcfd.cpp:185-199, kernels.cpp:365)
    SKB_TRY(eval_on_device(ctx, d, SKB_STOKESLET, kRaw, d_forces, 0.0, d_vel, accumulate, fl->cur, false,
                           &fl->launches, nullptr, 1.0 / eta));
    fl->pairs += fl->n_fib * d.n_trg;
    if (!subtract_self)
        return SKB_OK;
    if (!d.src[SKB_STOKESLET].excl && d.n_trg < node_end - node_begin)
        return set_error(SKB_ERR_INVALID, "fiber flow with subtract_self needs the fiber nodes as the first "
                                          "%lld targets (n_trg = %lld)", node_end - node_begin, d.n_trg);
    return fiber_self_term(fl, d, d.src[SKB_STOKESLET].f_cur, eta, d_vel, node_begin, node_end);
}

// mode kNormalDensity: d_density is the density, f_dl = 2 eta n (x) rho is formed on the device; kPacked: d_density
// holds the packed sym6 strengths already
static int periphery_dev(skb_flow *fl, skb_ctx *ctx, StrengthMode mode, const double *d_density, double eta,
                         double *d_vel, int accumulate) {
    DeviceState &d = ctx->devs[0];
    if (d.n_trg == 0)
        return SKB_OK;
    if (fl->n_shell == 0) { // periphery.cpp:57-58
        if (!accumulate)
            CUDA_TRY(cudaMemsetAsync(d_vel, 0, (size_t)d.n_trg * 24, fl->cur));
        return SKB_OK;
    }
    // stresslet, / eta  (periphery.cpp:68-74, kernels.cpp:358)
    SKB_TRY(eval_on_device(ctx, d, SKB_STRESSLET, mode, d_density, 2.0 * eta, d_vel, accumulate, fl->cur, false,
                           &fl->launches, nullptr, 1.0 / eta));
    fl->pairs += fl->n_shell * d.n_trg;
    return SKB_OK;
}

static int bodies_dev(skb_flow *fl, skb_ctx *ctx, const double *d_density, const double *d_force,
                      const double *d_torque, double eta, double *d_vel, int accumulate) {
    DeviceState &d = ctx->devs[0];
    if (d.n_trg == 0)
        return SKB_OK;
    if (fl->n_bodies == 0) { // body_container.cpp:273-276
        if (!accumulate)
            CUDA_TRY(cudaMemsetAsync(d_vel, 0, (size_t)d.n_trg * 24, fl->cur));
        return SKB_OK;
    }
    // stresslet of the surface nodes (body_container.cpp:296-305)
    SKB_TRY(eval_on_device(ctx, d, SKB_STRESSLET, kNormalDensity, d_density, 2.0 * eta, d_vel, accumulate, fl->cur,
                           false, &fl->launches, nullptr, 1.0 / eta));
    // Stokeslet of the net forces at the centres (:327)
    SKB_TRY(eval_on_device(ctx, d, SKB_STOKESLET, kRaw, d_force, 0.0, d_vel, 1, fl->cur, false, &fl->launches,
                           nullptr, 1.0 / eta));
    // rotlet of the net torques at the centres (:335, kernels.cpp:206-242)
    const int bs = 128;
    rotlet_add_kernel<<<(unsigned)((d.n_trg + bs - 1) / bs), bs, 0, fl->cur>>>(
        (const double *)fl->centers.ptr, d_torque, fl->n_bodies, (const double *)d.r_trg.ptr, d.n_trg,
        1.0 / (8.0 * M_PI * eta), kReg * kReg, kEps * kEps, d_vel);
    fl->pairs += (fl->n_body + 2 * (long long)fl->n_bodies) * d.n_trg;
    return launched(fl, 1);
}

// nothing to copy for an empty or absent (NULL) input
static int upload(skb_flow *fl, DevBuf &buf, const double *h, size_t n_doubles) {
    if (n_doubles == 0 || !h)
        return SKB_OK;
    SKB_TRY(buf.ensure(n_doubles * 8));
    CUDA_TRY(cudaMemcpyAsync(buf.ptr, h, n_doubles * 8, cudaMemcpyHostToDevice, fl->stream));
    return SKB_OK;
}

static int set_targets_cached(skb_ctx *ctx, TargetCache &tc, const double *r_trg, long long n_trg) {
    if (tc.same(r_trg, n_trg) && ctx->n_trg == n_trg)
        return SKB_OK;
    SKB_TRY(skb_set_targets(ctx, r_trg, n_trg));
    tc.store(r_trg, n_trg);
    return SKB_OK;
}

static void split_forces_torques(const double *ft, int n_bodies, std::vector<double> &f, std::vector<double> &t) {
    f.resize(3 * (size_t)n_bodies);
    t.resize(3 * (size_t)n_bodies);
    for (int b = 0; b < n_bodies; ++b)
        for (int k = 0; k < 3; ++k) {
            f[3 * b + k] = ft[6 * b + k];     // forces_torques.block(0,0,3,n)  body_container.cpp:134
            t[3 * b + k] = ft[6 * b + 3 + k]; // forces_torques.block(3,0,3,n)
        }
}

// host strengths of one flow call: fiber forces and periphery density (3 per node), body densities (3 per node), net
// body forces and torques (3 per body, split_forces_torques)
struct HostStrengths {
    const double *ff, *sd, *bd, *f, *t;
};
static size_t n_strengths(const skb_flow *fl) {
    return (size_t)(fl->n_fib + fl->n_shell + fl->n_body) * 3 + 6 * (size_t)fl->n_bodies;
}
static int upload_strengths(skb_flow *fl, const HostStrengths &in) {
    SKB_TRY(upload(fl, fl->in_fib, in.ff, (size_t)fl->n_fib * 3));
    SKB_TRY(upload(fl, fl->in_shell, in.sd, (size_t)fl->n_shell * 3));
    SKB_TRY(upload(fl, fl->in_body, in.bd, (size_t)fl->n_body * 3));
    SKB_TRY(upload(fl, fl->in_force, in.f, 3 * (size_t)fl->n_bodies));
    SKB_TRY(upload(fl, fl->in_torque, in.t, 3 * (size_t)fl->n_bodies));
    return SKB_OK;
}


// ---- CUDA-graph helpers ----------------------------------------------------------------------------------------
static constexpr size_t kGraphMaxBytes = 512 * 1024; // strengths + velocities of one call; beyond this the copies
                                                     // and kernels dwarf the launch gaps and the plain path is used
static unsigned long long mix_key(unsigned long long h, unsigned long long v) {
    h ^= v + 0x9e3779b97f4a7c15ULL + (h << 6) + (h >> 2);
    return h;
}
static unsigned long long dbl_bits(double x) {
    unsigned long long b;
    std::memcpy(&b, &x, 8);
    return b;
}
static int ensure_stage(skb_flow *fl, size_t n_doubles) {
    if (n_doubles <= fl->h_stage_cap)
        return SKB_OK;
    if (fl->h_stage)
        cudaFreeHost(fl->h_stage);
    fl->h_stage = nullptr;
    fl->h_stage_cap = 0;
    fl->g_matvec.reset(); // graphs hold the old staging addresses
    fl->g_vat.reset();
    CUDA_TRY(cudaMallocHost((void **)&fl->h_stage, (n_doubles + 64) * 8));
    fl->h_stage_cap = n_doubles + 64;
    return SKB_OK;
}

// Copy a graphed call's strengths into the pinned stage, laid out as [fiber forces | periphery density | body densities
// | body forces | body torques | n_out output values]; *staged points at the copies, *h_out at the output values.
static int fill_stage(skb_flow *fl, const HostStrengths &in, size_t n_out, HostStrengths *staged, double **h_out) {
    const size_t nf = (size_t)fl->n_fib * 3, ns = (size_t)fl->n_shell * 3, nb = (size_t)fl->n_body * 3,
                 nft = 3 * (size_t)fl->n_bodies;
    SKB_TRY(ensure_stage(fl, n_strengths(fl) + n_out));
    double *h_ff = fl->h_stage, *h_sd = h_ff + nf, *h_bd = h_sd + ns, *h_f = h_bd + nb, *h_t = h_f + nft;
    if (nf) std::memcpy(h_ff, in.ff, nf * 8);
    if (ns) std::memcpy(h_sd, in.sd, ns * 8);
    if (nb) std::memcpy(h_bd, in.bd, nb * 8);
    if (nft) std::memcpy(h_f, in.f, nft * 8);
    if (nft) std::memcpy(h_t, in.t, nft * 8);
    *staged = HostStrengths{h_ff, h_sd, h_bd, h_f, h_t};
    *h_out = h_t + nft;
    return SKB_OK;
}

// every device address a captured sequence may bake in: a reallocation anywhere invalidates the graph
static unsigned long long buffer_key(const skb_flow *fl, int which) {
    unsigned long long h = 0x1234567ULL;
    const DevBuf *bufs[] = {&fl->in_fib, &fl->in_shell, &fl->in_body, &fl->in_force, &fl->in_torque, &fl->vel,
                            &fl->tmp,    &fl->pt_pos,   &fl->pt_force, &fl->pt_torque, &fl->centers, &fl->r_fib};
    for (const DevBuf *b : bufs)
        h = mix_key(h, (unsigned long long)(uintptr_t)b->ptr);
    const skb_ctx *ctxs[] = {fl->fib[which], fl->shell[which], fl->body[which]};
    for (const skb_ctx *c : ctxs) {
        const DeviceState &d = c->devs[0];
        h = mix_key(h, (unsigned long long)(uintptr_t)d.r_trg.ptr);
        h = mix_key(h, (unsigned long long)(uintptr_t)d.partial.ptr);
        for (int k = 0; k < 2; ++k) {
            h = mix_key(h, (unsigned long long)(uintptr_t)d.src[k].f_packed.ptr);
            h = mix_key(h, (unsigned long long)(uintptr_t)d.src[k].r.ptr);
        }
    }
    return h;
}

// Run `body` (asynchronous work on fl->stream, fixed addresses only) either directly, as a capture followed by a
// replay, or as a replay of the cached graph.  First call with a key: direct (it also warms every buffer); second
// call with the same key: captured; afterwards: one cudaGraphLaunch per call.
template <class Body> static int run_graphed(skb_flow *fl, skb_flow::GraphSlot &slot, unsigned long long key, Body body) {
    if (slot.exec && slot.key == key) {
        CUDA_TRY(cudaGraphLaunch(slot.exec, fl->stream));
        count_launch(slot.launches);
        fl->launches = slot.launches;
        fl->pairs = slot.pairs;
        return SKB_OK;
    }
    if (slot.seen == key && fl->graphs_enabled) {
        if (slot.exec) {
            cudaGraphExecDestroy(slot.exec);
            slot.exec = nullptr;
        }
        cudaGraph_t graph = nullptr;
        const long long before = launch_count();
        CUDA_TRY(cudaStreamBeginCapture(fl->stream, cudaStreamCaptureModeThreadLocal));
        const int rc = body();
        cudaError_t e = cudaStreamEndCapture(fl->stream, &graph);
        count_launch((int)(before - launch_count())); // nothing was launched while capturing
        if (rc == SKB_OK && e == cudaSuccess && graph &&
            cudaGraphInstantiate(&slot.exec, graph, nullptr, nullptr, 0) == cudaSuccess) {
            cudaGraphDestroy(graph);
            slot.key = key;
            slot.launches = fl->launches;
            slot.pairs = fl->pairs;
            CUDA_TRY(cudaGraphLaunch(slot.exec, fl->stream));
            count_launch(slot.launches);
            return SKB_OK;
        }
        if (graph)
            cudaGraphDestroy(graph);
        (void)cudaGetLastError();
        slot.exec = nullptr;
        fl->graphs_enabled = false; // capture is not possible in this process: stay on the direct path
        fl->launches = 0;
        fl->pairs = 0;
    }
    slot.seen = key;
    return body();
}

// ---- call scaffolding ------------------------------------------------------------------------------------------
// every evaluating entry point: on the flow's device, launch and pair counts of this call from zero
static int begin_call(skb_flow *fl) {
    CUDA_TRY(cudaSetDevice(fl->dev));
    fl->launches = 0;
    fl->pairs = 0;
    return SKB_OK;
}
// *_device calls run on the caller's stream and take no times
static int device_call_finish(skb_flow *fl) {
    fl->stats.device_ms = fl->stats.total_ms = 0;
    fl->stats.n_pairs = fl->pairs;
    fl->stats.launches = fl->launches;
    return SKB_OK;
}
// Host-pointer calls run on fl->stream: total_ms spans evt0 (host_call_start, before the uploads) to evt1
// (host_call_finish, after the downloads); device_ms spans ev0 to ev1, which the call records around its device work.
static int host_call_start(skb_flow *fl) {
    fl->cur = fl->stream;
    CUDA_TRY(cudaEventRecord(fl->evt0, fl->stream));
    return SKB_OK;
}
static int host_call_finish(skb_flow *fl) {
    CUDA_TRY(cudaEventRecord(fl->evt1, fl->stream));
    CUDA_TRY(cudaStreamSynchronize(fl->stream));
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, fl->ev0, fl->ev1);
    cudaEventElapsedTime(&b, fl->evt0, fl->evt1);
    SKB_TRY(device_call_finish(fl));
    fl->stats.device_ms = a;
    fl->stats.total_ms = b;
    return SKB_OK;
}

// resolve the target window / ranges into fiber, shell and body pieces and (re)build the matvec target lists
static int prepare_matvec_targets(skb_flow *fl) {
    const long long nf = fl->n_fib, ns = fl->n_shell, nb = fl->n_body, n_all = nf + ns + nb;
    if (!fl->mv_dirty)
        return SKB_OK;
    auto clampi = [](long long x, long long lo, long long hi) { return std::min(std::max(x, lo), hi); };
    if (fl->use_ranges) {
        const long long f0 = clampi(fl->rq_f0, 0, fl->n_fibers), f1 = clampi(fl->rq_f1, f0, fl->n_fibers);
        fl->fa = fl->n_fibers ? fl->h_fiber_off[(size_t)f0] : 0;
        fl->fb = fl->n_fibers ? fl->h_fiber_off[(size_t)f1] : 0;
        fl->sa = clampi(fl->rq_s0, 0, ns);
        fl->sb = clampi(fl->rq_s1, fl->sa, ns);
        fl->ba = clampi(fl->rq_b0, 0, nb);
        fl->bb = clampi(fl->rq_b1, fl->ba, nb);
    } else {
        long long w0 = fl->win_begin, w1 = fl->win_end < 0 ? n_all : fl->win_end;
        w0 = clampi(w0, 0, n_all);
        w1 = clampi(w1, w0, n_all);
        fl->fa = clampi(w0, 0, nf);
        fl->fb = clampi(w1, 0, nf);
        fl->sa = clampi(w0 - nf, 0, ns);
        fl->sb = clampi(w1 - nf, 0, ns);
        fl->ba = clampi(w0 - nf - ns, 0, nb);
        fl->bb = clampi(w1 - nf - ns, 0, nb);
    }
    const long long n_fw = fl->fb - fl->fa, n_sw = fl->sb - fl->sa, n_bw = fl->bb - fl->ba;
    fl->n_win = n_fw + n_sw + n_bw;
    const bool grouped = fl->grp.size > 1;
    if (grouped) {
        if (!fl->use_ranges)
            return set_error(SKB_ERR_STATE, "group member: call skb_flow_set_target_ranges (own fibers / periphery rows / "
                                            "body rows) before the first matvec");
        if (fl->grp.n_fib != nf || fl->grp.n_shell != ns)
            return set_error(SKB_ERR_STATE, "group member: the geometry changed size since skb_flow_group_init "
                                            "(%lld/%lld fiber, %lld/%lld periphery nodes); re-initialise the group",
                             nf, fl->grp.n_fib, ns, fl->grp.n_shell);
        // fiber rows through the symmetric block rows of this member (partial sums, pulled together afterwards) when
        // the self-interaction is big enough for that kernel; otherwise the member's own rows with the plain kernel
        fl->grp.use_sym = nf >= 2LL * sym_block_nodes();
    }
    // fiber <-> periphery pairs in one pass (cross_kernels.cuh) when both classes are big enough to matter and the
    // symmetric kernel carries the fiber rows (so that the fiber evaluator's remaining targets are the body rows only)
    static const int cross_env = [] {
        const char *e = getenv("SKB_CROSS");
        return e ? atoi(e) : -1;
    }();
    const int cmode = fl->cross_mode >= 0 ? fl->cross_mode : cross_env;
    const bool sym_rows = grouped ? fl->grp.use_sym
                                  : (fl->fa == 0 && fl->fb == nf && fl->sa == 0 && fl->sb == ns &&
                                     nf >= (cmode == 1 ? 2LL * sym_block_nodes() : 4096));
    fl->use_cross = cmode != 0 && sym_rows && n_fw > 0 && ns >= (cmode == 1 ? 1 : 256);
    // target lists of apply_matvec: r_all = [fibers | shell | bodies] (system.cpp:284-291),
    // r_fibbody = [fibers | bodies] (system.cpp:301-303), both restricted to this rank's pieces
    std::vector<double> r_win, r_fb;
    r_win.reserve((size_t)fl->n_win * 3);
    r_win.insert(r_win.end(), fl->h_r_fib.begin() + 3 * fl->fa, fl->h_r_fib.begin() + 3 * fl->fb);
    r_win.insert(r_win.end(), fl->h_r_shell.begin() + 3 * fl->sa, fl->h_r_shell.begin() + 3 * fl->sb);
    r_win.insert(r_win.end(), fl->h_r_body.begin() + 3 * fl->ba, fl->h_r_body.begin() + 3 * fl->bb);
    if (!fl->use_cross)
        r_fb.insert(r_fb.end(), fl->h_r_fib.begin() + 3 * fl->fa, fl->h_r_fib.begin() + 3 * fl->fb);
    r_fb.insert(r_fb.end(), fl->h_r_body.begin() + 3 * fl->ba, fl->h_r_body.begin() + 3 * fl->bb);
    if (grouped && fl->grp.use_sym) {
        // fiber sources meet [ALL fiber nodes | own shell rows | own body rows]; with the cross kernel the periphery
        // rows are not targets of this evaluator
        std::vector<double> r_sym;
        r_sym.reserve((size_t)(nf + n_sw + n_bw) * 3);
        r_sym.insert(r_sym.end(), fl->h_r_fib.begin(), fl->h_r_fib.end());
        if (!fl->use_cross)
            r_sym.insert(r_sym.end(), fl->h_r_shell.begin() + 3 * fl->sa, fl->h_r_shell.begin() + 3 * fl->sb);
        r_sym.insert(r_sym.end(), fl->h_r_body.begin() + 3 * fl->ba, fl->h_r_body.begin() + 3 * fl->bb);
        SKB_TRY(skb_ctx_set_symmetric(fl->fib[1], 1));
        SKB_TRY(skb_ctx_set_sym_partition(fl->fib[1], fl->grp.rank, fl->grp.size));
        SKB_TRY(skb_set_targets(fl->fib[1], r_sym.data(), (long long)r_sym.size() / 3));
    } else if (fl->use_cross) {
        std::vector<double> r_fibbody(fl->h_r_fib.begin() + 3 * fl->fa, fl->h_r_fib.begin() + 3 * fl->fb);
        r_fibbody.insert(r_fibbody.end(), fl->h_r_body.begin() + 3 * fl->ba, fl->h_r_body.begin() + 3 * fl->bb);
        SKB_TRY(skb_ctx_set_sym_partition(fl->fib[1], 0, 1));
        SKB_TRY(skb_set_targets(fl->fib[1], r_fibbody.data(), (long long)r_fibbody.size() / 3));
    } else {
        SKB_TRY(skb_ctx_set_sym_partition(fl->fib[1], 0, 1));
        SKB_TRY(skb_set_targets(fl->fib[1], r_win.data(), fl->n_win));
    }
    SKB_TRY(skb_set_targets(fl->body[1], r_win.data(), fl->n_win));
    SKB_TRY(skb_set_targets(fl->shell[1], r_fb.data(), (long long)r_fb.size() / 3));
    const bool all_fibers_lead = (fl->fa == 0 && fl->fb == nf) || (grouped && fl->grp.use_sym);
    if (fl->self_excl && fl->n_fib > 0) {
        if (!all_fibers_lead)
            return set_error(SKB_ERR_INVALID, "skb_flow_set_self_exclusion needs all fiber nodes as the leading matvec "
                                              "targets (no target window / ranges that cut the fiber rows)");
        std::vector<int32_t> ids((size_t)nf);
        for (int f = 0; f < fl->n_fibers; ++f)
            for (long long i = fl->h_fiber_off[(size_t)f]; i < fl->h_fiber_off[(size_t)f + 1]; ++i)
                ids[(size_t)i] = f;
        SKB_TRY(skb_set_source_exclusion_ids(fl->fib[1], ids.data(), nf));
    } else {
        SKB_TRY(skb_set_source_exclusion_ids(fl->fib[1], nullptr, 0));
    }
    fl->mv_dirty = false;
    return SKB_OK;
}

// ---- group exchange steps (group_kernels.cuh) on fl->cur ---------------------------------------------------------
// The pending dense product of apply_matvec_core goes out on the side stream, ordered after everything on fl->cur so far
// (its input is complete), and runs beside whatever fl->cur launches next.  The side stream has the highest priority:
// its 148 one-warp CTAs are placed before the pair kernel's CTAs fill the SMs.
static int overlap_buffers(skb_flow *fl, long long n_rows) {
    skb_flow::Overlap &B = fl->bg;
    if (!B.stream) {
        int lo = 0, hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&B.stream, cudaStreamNonBlocking, hi));
        CUDA_TRY(cudaEventCreateWithFlags(&B.fork, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&B.join, cudaEventDisableTiming));
        // nothing may be loaded lazily later, while a group member on this device spins on a flag
        SKB_TRY(dense_stream_preload(fl->dev));
        cudaFuncAttributes fa;
        CUDA_TRY(cudaFuncGetAttributes(&fa, add_out_kernel));
    }
    SKB_TRY(B.y.ensure((size_t)n_rows * 8 + 8));
    return SKB_OK;
}
static int overlap_launch(skb_flow *fl) {
    skb_flow::Overlap &B = fl->bg;
    if (!B.dn || B.launched)
        return SKB_OK;
    CUDA_TRY(cudaEventRecord(B.fork, fl->cur));
    CUDA_TRY(cudaStreamWaitEvent(B.stream, B.fork, 0));
    SKB_TRY(skb_dense_apply_background_device(B.dn, SKB_DENSE_STRESSLET_PLUS_COMPLEMENTARY, B.d_x, (double *)B.y.ptr,
                                              B.stream));
    CUDA_TRY(cudaEventRecord(B.join, B.stream));
    B.launched = true;
    fl->launches += 1;
    return SKB_OK;
}

static int group_flag(skb_flow *fl, int phase, bool do_signal, bool do_wait) {
    skb_flow::Group &G = fl->grp;
    if (G.dry)
        return SKB_OK;
    GroupFlagArgs a;
    for (int m = 0; m < G.size; ++m)
        a.flags[m] = G.at<unsigned long long>(m, G.off_flags);
    a.rank = G.rank;
    a.size = G.size;
    a.phase = phase;
    a.epoch = G.epoch;
    a.do_signal = do_signal;
    a.do_wait = do_wait;
    a.timeout_cycles = 20ULL * 1000 * 1000 * 1000; // ~10 s at 2 GHz
    group_flag_kernel<<<1, 32, 0, fl->cur>>>(a);
    return launched(fl, 1);
}

// window addresses at `off` of the members a push or pull reaches -- every member, or only this one in a dry run;
// returns their count
template <class T> static int member_windows(const skb_flow::Group &G, size_t off, T **out) {
    const int n = G.dry ? 1 : G.size;
    for (int m = 0; m < n; ++m)
        out[m] = G.at<double>(G.dry ? G.rank : m, off);
    return n;
}

// PULL: rows [first, first + n) of d_out += the members' partial sums at window offset `off` (reduce-scatter fused
// with the accumulation, members added in rank order)
static int group_pull(skb_flow *fl, size_t off, long long first, long long n, double *d_out) {
    GroupPullArgs a;
    a.size = member_windows(fl->grp, off, a.u_part);
    a.fa = first;
    a.n_f = n;
    a.v = d_out;
    a.accumulate = 1;
    group_pull_kernel<<<(unsigned)((3 * n + 255) / 256), 256, 0, fl->cur>>>(a);
    return launched(fl, 1);
}

// v_fibers, v_bodies += shell.flow(r_fibbody, x_shell, eta)   (system.cpp:304,313-315) at the own rows of d_v, with
// the periphery strengths d_s in `mode`.  The periphery evaluator's targets are [own fiber rows | own body rows], the
// body rows alone with the cross kernel (it does the fiber rows).  The flow lands in fl->tmp and is added into d_v;
// fib_unset: d_v's fiber rows hold nothing yet (a group's symmetric partial sums are pulled in later), so the flow is
// copied there instead -- zeros without a periphery.
static int periphery_into_rows(skb_flow *fl, StrengthMode mode, const double *d_s, double eta, double *d_v,
                               bool fib_unset) {
    const long long n_fw = fl->fb - fl->fa, n_sw = fl->sb - fl->sa, n_bw = fl->bb - fl->ba;
    const long long n_ft = fl->use_cross ? 0 : n_fw; // fiber rows among the evaluator's targets
    if (fl->n_shell > 0 && n_ft + n_bw > 0) {
        SKB_TRY(fl->tmp.ensure((size_t)(n_ft + n_bw) * 24 + 8));
        double *d_tmp = (double *)fl->tmp.ptr;
        SKB_TRY(periphery_dev(fl, fl->shell[1], mode, d_s, eta, d_tmp, 0));
        if (n_ft > 0 && fib_unset) {
            CUDA_TRY(cudaMemcpyAsync(d_v, d_tmp, (size_t)n_ft * 24, cudaMemcpyDeviceToDevice, fl->cur));
        } else if (n_ft > 0) {
            add_inplace_kernel<<<(unsigned)((3 * n_ft + 255) / 256), 256, 0, fl->cur>>>(d_v, d_tmp, 3 * n_ft);
            SKB_TRY(launched(fl, 1));
        }
        if (n_bw > 0) {
            add_inplace_kernel<<<(unsigned)((3 * n_bw + 255) / 256), 256, 0, fl->cur>>>(
                d_v + 3 * (n_fw + n_sw), d_tmp + 3 * n_ft, 3 * n_bw);
            SKB_TRY(launched(fl, 1));
        }
    } else if (n_ft > 0 && fib_unset) {
        CUDA_TRY(cudaMemsetAsync(d_v, 0, (size_t)n_ft * 24, fl->cur));
    }
    return SKB_OK;
}

// device-side matvec flow of a group member on fl->cur: d_ff / d_sd are the strengths of the OWN fibers / periphery
// rows, body inputs are complete on every member; d_v = [own fiber rows | own shell rows | own body rows] of v_all
static int matvec_core_group(skb_flow *fl, const double *d_ff, const double *d_sd, const double *d_bd, const double *d_f,
                             const double *d_t, double eta, double *d_v) {
    skb_flow::Group &G = fl->grp;
    if (!G.dry && !G.connected())
        return set_error(SKB_ERR_STATE, "group member %d: not all peers are connected (skb_flow_group_import / _connect)",
                         G.rank);
    const long long ns = fl->n_shell, nf = fl->n_fib;
    const long long n_fw = fl->fb - fl->fa, n_sw = fl->sb - fl->sa, n_bw = fl->bb - fl->ba;
    G.epoch += 1;
    const int par = (int)(G.epoch & 1);
    DeviceState &df = fl->fib[1]->devs[0];
    // 1. PUSH: pack own strengths once, store them into every member's window (pack + all-gather in one kernel)
    {
        GroupPushArgs a;
        a.fw = d_ff;
        a.weight = df.src[SKB_STOKESLET].has_weights ? (const double *)df.src[SKB_STOKESLET].weights.ptr : nullptr;
        a.fa = fl->fa;
        a.n_f = n_fw;
        a.density = d_sd;
        a.normal = ns ? (const double *)fl->shell[1]->devs[0].src[SKB_STRESSLET].normals.ptr : nullptr;
        a.sa = fl->sa;
        a.n_s = n_sw;
        a.two_eta = 2.0 * eta;
        a.size = member_windows(G, G.off_fsl[par], a.f_sl);
        member_windows(G, G.off_fshell[par], a.f_shell);
        member_windows(G, G.off_xshell[par], a.x_shell);
        const long long work = 3 * n_fw + n_sw;
        if (work > 0) {
            const unsigned nblk = (unsigned)std::min<long long>((work + 255) / 256, 4LL * df.info.num_sms);
            group_push_kernel<<<nblk, 256, 0, fl->cur>>>(a);
            SKB_TRY(launched(fl, 1));
        }
    }
    // 2. every member's strengths have landed here
    SKB_TRY(group_flag(fl, 0, true, true));
    SKB_TRY(overlap_launch(fl)); // (x_shell is complete in the window from here on)
    const double *f_sl = G.at<double>(G.rank, G.off_fsl[par]);
    const double *f_shell = G.at<double>(G.rank, G.off_fshell[par]);
    double *u_part = G.at<double>(G.rank, G.off_upart);
    // 3. v = fc.flow(r_all, fw, eta)  (system.cpp:299): own block rows of the symmetric fiber-fiber interaction
    //    (partial sums for ALL fiber nodes -> u_part) + own shell / body rows (complete -> d_v)
    if (fl->n_fibers > 0 && df.n_trg > 0) {
        if (G.use_sym) {
            SKB_TRY(fl->scratch_u.ensure((size_t)df.n_trg * 24));
            EvalOpts o;
            o.d_u_sym = u_part;
            o.sym_accumulate = 0;
            o.d_u_rem = fl->use_cross ? d_v + 3 * (n_fw + n_sw) : d_v + 3 * n_fw; // cross: body rows only
            SKB_TRY(eval_on_device(fl->fib[1], df, SKB_STOKESLET, kPacked, f_sl, 0.0, (double *)fl->scratch_u.ptr, 0,
                                   fl->cur, false, &fl->launches, nullptr, 1.0 / eta, o));
            if (!fl->fib[1]->last_was_sym)
                return set_error(SKB_ERR_STATE, "group member %d: the symmetric kernel declined (memory for the reverse "
                                                "partials?); lower SKB_SYM_MAX_BYTES pressure or use fewer nodes per GPU",
                                 G.rank);
            fl->pairs += nf * nf / G.size + nf * ((fl->use_cross ? 0 : n_sw) + n_bw);
            if (fl->use_cross && ns > 0) {
                // own fibers x ALL periphery nodes in one pass: stresslet sums at the own fiber rows (complete) and
                // this member's partial Stokeslet sums at every periphery row (pulled together after flag B)
                DeviceState &dsh = fl->shell[1]->devs[0];
                const SourceSet &sf = df.src[SKB_STOKESLET], &ss = dsh.src[SKB_STRESSLET];
                SKB_TRY(cross_eval(fl->cross, df.info, (const double *)sf.r.ptr, f_sl, fl->fa, n_fw,
                                   (const double *)ss.r.ptr, f_shell, ns, ss.n_pad, -3.0 / (8.0 * M_PI * eta),
                                   1.0 / (8.0 * M_PI * eta), d_v, 0, G.at<double>(G.rank, G.off_upart_shell), 0, fl->cur,
                                   &fl->launches));
                fl->pairs += 2 * n_fw * ns;
            }
            SKB_TRY(group_flag(fl, 1, true, false)); // my partial sums are complete
        } else {
            SKB_TRY(eval_on_device(fl->fib[1], df, SKB_STOKESLET, kPacked, f_sl, 0.0, d_v, 0, fl->cur, false,
                                   &fl->launches, nullptr, 1.0 / eta));
            fl->pairs += nf * df.n_trg;
        }
    } else if (fl->n_win > 0) {
        CUDA_TRY(cudaMemsetAsync(d_v, 0, (size_t)fl->n_win * 24, fl->cur));
    }
    // d_v's fiber rows are not complete yet.  (use_cross implies the symmetric rows, own fibers and a periphery, so the
    // cross kernel ran above and wrote the own fiber rows.)
    const bool fib_rows_pending = G.use_sym && fl->n_fibers > 0;
    // 4. v_fibers, v_bodies += shell.flow(r_fibbody, x_shell, eta)   (system.cpp:304,313-315)
    if (fl->use_cross && n_sw > 0) // own periphery rows: body flow first, the members' Stokeslet partials pulled in below
        CUDA_TRY(cudaMemsetAsync(d_v + 3 * n_fw, 0, (size_t)n_sw * 24, fl->cur));
    SKB_TRY(periphery_into_rows(fl, kPacked, f_shell, eta, d_v, fib_rows_pending));
    // 5. v_all += bc.flow(r_all, x_bodies, body_link_conditions, eta)     (system.cpp:316)
    SKB_TRY(bodies_dev(fl, fl->body[1], d_bd, d_f, d_t, eta, d_v, 1));
    // 6. PULL: own fiber rows += sum over the members' partial sums
    if (fib_rows_pending) {
        SKB_TRY(group_flag(fl, 1, false, true));
        if (n_fw > 0)
            SKB_TRY(group_pull(fl, G.off_upart, fl->fa, n_fw, d_v));
        if (fl->use_cross && n_sw > 0) // own periphery rows += the members' Stokeslet partials
            SKB_TRY(group_pull(fl, G.off_upart_shell, fl->sa, n_sw, d_v + 3 * n_fw));
    }
    // 7. self term of the own fibers
    if (n_fw > 0)
        SKB_TRY(fiber_self_term(fl, df, f_sl, eta, d_v, fl->fa, fl->fb));
    return SKB_OK;
}

// The same with the fiber <-> periphery pairs in one geometry pass (cross_kernels.cuh): whole system on this device.
//   fiber evaluator targets  = [fibers | bodies]   (symmetric fiber-fiber block + the body rows)
//   cross kernel             : stresslet of every periphery node at the fiber nodes, Stokeslet of every fiber node at
//                              the periphery nodes (system.cpp:299 and :304,313-315 from one pass over the pairs)
//   periphery evaluator      = [bodies] only
static int matvec_core_cross(skb_flow *fl, const double *d_ff, const double *d_sd, const double *d_bd, const double *d_f,
                             const double *d_t, double eta, double *d_v) {
    const long long ns = fl->n_shell, nf = fl->n_fib;
    const long long n_fw = fl->fb - fl->fa, n_sw = fl->sb - fl->sa, n_bw = fl->bb - fl->ba; // == nf, ns, nb here
    DeviceState &df = fl->fib[1]->devs[0];
    DeviceState &dsh = fl->shell[1]->devs[0];
    double *d_v_body = d_v + 3 * (n_fw + n_sw);
    // fc.flow at [fibers | bodies]: the symmetric kernel writes the fiber rows, the plain kernel the body rows.  Should the
    // symmetric path decline (memory), everything lands contiguously in the scratch buffer and is moved into place.
    SKB_TRY(fl->scratch_u.ensure((size_t)df.n_trg * 24 + 8));
    EvalOpts o;
    o.d_u_sym = d_v;
    o.d_u_rem = d_v_body;
    SKB_TRY(eval_on_device(fl->fib[1], df, SKB_STOKESLET, kRaw, d_ff, 0.0, (double *)fl->scratch_u.ptr, 0, fl->cur, false,
                           &fl->launches, nullptr, 1.0 / eta, o));
    if (!fl->fib[1]->last_was_sym) {
        CUDA_TRY(cudaMemcpyAsync(d_v, fl->scratch_u.ptr, (size_t)n_fw * 24, cudaMemcpyDeviceToDevice, fl->cur));
        if (n_bw > 0)
            CUDA_TRY(cudaMemcpyAsync(d_v_body, (const double *)fl->scratch_u.ptr + 3 * n_fw, (size_t)n_bw * 24,
                                     cudaMemcpyDeviceToDevice, fl->cur));
    }
    fl->pairs += nf * (n_fw + n_bw);
    SKB_TRY(fiber_self_term(fl, df, df.src[SKB_STOKESLET].f_cur, eta, d_v, fl->fa, fl->fb));
    // periphery strengths 2 eta n (x) rho -> sym6 (periphery.cpp:68-71), once for both uses
    SKB_TRY(pack_on_device(dsh, SKB_STRESSLET, kNormalDensity, d_sd, 2.0 * eta, fl->cur, &fl->launches));
    const SourceSet &sf = df.src[SKB_STOKESLET], &ss = dsh.src[SKB_STRESSLET];
    SKB_TRY(cross_eval(fl->cross, df.info, (const double *)sf.r.ptr, sf.f_cur, fl->fa, n_fw, (const double *)ss.r.ptr,
                       ss.f_cur, ns, ss.n_pad, -3.0 / (8.0 * M_PI * eta), 1.0 / (8.0 * M_PI * eta), d_v, 1,
                       d_v + 3 * n_fw, 0, fl->cur, &fl->launches));
    fl->pairs += 2 * n_fw * ns;
    // periphery -> body rows (system.cpp:313-315)
    SKB_TRY(periphery_into_rows(fl, kPacked, ss.f_cur, eta, d_v, false));
    // v_all += bc.flow(r_all, x_bodies, body_link_conditions, eta)     system.cpp:316
    SKB_TRY(bodies_dev(fl, fl->body[1], d_bd, d_f, d_t, eta, d_v, 1));
    return SKB_OK;
}

// device-side matvec flow on fl->cur: all strengths resident, d_v = window rows of v_all
static int matvec_core(skb_flow *fl, const double *d_ff, const double *d_sd, const double *d_bd, const double *d_f,
                       const double *d_t, double eta, double *d_v) {
    if (fl->grp.size > 1)
        return matvec_core_group(fl, d_ff, d_sd, d_bd, d_f, d_t, eta, d_v);
    const long long n_fw = fl->fb - fl->fa;
    if (fl->n_win == 0)
        return SKB_OK;
    SKB_TRY(overlap_launch(fl));
    if (fl->use_cross)
        return matvec_core_cross(fl, d_ff, d_sd, d_bd, d_f, d_t, eta, d_v);
    // v_all = fc.flow(r_all, fw, eta)                                  system.cpp:299
    // (this rank's fiber rows come first, so the self term applies to targets [0, n_fw) of its list)
    SKB_TRY(fibers_dev(fl, fl->fib[1], d_ff, eta, n_fw > 0, d_v, 0, fl->fa, fl->fb));
    // v_fibers, v_bodies += shell.flow(r_fibbody, x_shell, eta)         system.cpp:304,313-315
    SKB_TRY(periphery_into_rows(fl, kNormalDensity, d_sd, eta, d_v, false));
    // v_all += bc.flow(r_all, x_bodies, body_link_conditions, eta)     system.cpp:316
    SKB_TRY(bodies_dev(fl, fl->body[1], d_bd, d_f, d_t, eta, d_v, 1));
    return SKB_OK;
}

static void group_release(skb_flow *fl) {
    skb_flow::Group &G = fl->grp;
    cudaSetDevice(fl->dev);
    for (int m = 0; m < G.size; ++m)
        if (m != G.rank && G.peer[m] && G.peer_ipc[m])
            cudaIpcCloseMemHandle(G.peer[m]);
    if (G.window)
        cudaFree(G.window);
    G = skb_flow::Group();
}

static int need_ops(const skb_flow *fl, const char *who) {
    if (!fl->ops_ready)
        return set_error(SKB_ERR_INVALID, "%s: call skb_flow_set_fiber_operators after skb_flow_set_fibers / "
                                          "skb_flow_set_fiber_class first", who);
    return SKB_OK;
}

// y = A_^-1 x per fiber: FiberContainerFiniteDifference::apply_preconditioner (fcfd.cpp:331-339) with the LU solve
// replaced by a GEMV over the explicit inverse (same shapes and item list as A_); on fl->cur
static int fiber_precond_dev(skb_flow *fl, const double *d_x, double *d_y) {
    if (fl->n_items_A == 0)
        return SKB_OK;
    fiber_gemv_kernel<0><<<fl->n_items_A, kFiberGemvThreads, fl->gemv_smem, fl->cur>>>(
        (const FiberGemvItem *)fl->items_A.ptr, (const double *)fl->op_Ainv.ptr, d_x, d_y, FiberVelArgs{});
    return launched(fl, 1);
}
// (the three fiber_gemv_kernel modes are instantiated in mode order: 0 here, then 1 and 2)

// fw = force_operator_ * x per fiber, scattered to 3 x N_f (fcfd.cpp:272-287); on fl->cur
static int fiber_force_dev(skb_flow *fl, const double *d_x, double *d_fw) {
    if (fl->n_items_F == 0)
        return SKB_OK;
    fiber_gemv_kernel<1><<<fl->n_items_F, kFiberGemvThreads, fl->gemv_smem, fl->cur>>>(
        (const FiberGemvItem *)fl->items_F.ptr, (const double *)fl->op_F.ptr, d_x, d_fw, FiberVelArgs{});
    return launched(fl, 1);
}

// res = A_ x - P_downsample_bc vT(v) + xs_vT + y_BC per fiber (ffd.cpp:276-312), one launch; on fl->cur
static int fiber_matvec_dev(skb_flow *fl, const double *d_x, const double *d_v, const double *d_vb, double *d_res) {
    if (fl->n_items_A == 0)
        return SKB_OK;
    FiberVelArgs va;
    va.xs = (const double *)fl->op_xs.ptr;
    va.v = d_v;
    va.length_prev = (const double *)fl->op_len.ptr;
    va.plus_velocity = (const int *)fl->op_plus.ptr;
    va.class_mats = (const double *)fl->op_class.ptr;
    va.class_D = (const long long *)fl->op_classD.ptr;
    va.class_P = (const long long *)fl->op_classP.ptr;
    va.row_range = (const int2 *)fl->op_ranges.ptr;
    va.class_R = (const long long *)fl->op_classR.ptr;
    va.v_boundary = d_vb;
    fiber_gemv_kernel<2><<<fl->n_items_A, kFiberGemvThreads, fl->gemv_smem, fl->cur>>>(
        (const FiberGemvItem *)fl->items_A.ptr, (const double *)fl->op_A.ptr, d_x, d_res, va);
    return launched(fl, 1);
}

static int need_precond(const skb_flow *fl, const char *who) {
    SKB_TRY(need_ops(fl, who));
    if (fl->precond_gen != fl->ops_gen)
        return set_error(SKB_ERR_INVALID, "%s: call skb_flow_set_fiber_preconditioner after "
                                          "skb_flow_set_fiber_operators first", who);
    return SKB_OK;
}

// System::apply_matvec (system.cpp:298-319) on fl->cur, everything device resident.  Inputs are the OWN slices of a
// group member (all of them without a group): d_x 4 per own fiber node, d_xs 3 per own periphery row, body inputs
// complete, d_link 7 per own fiber or NULL.  Outputs: d_res_fib 4 per own node, d_out_shell 3 per own periphery row
// (res_shell when dn != NULL, else v_shell), d_v_bodies 3 per own body row; any of them may be NULL when empty.
static int apply_matvec_core(skb_flow *fl, skb_dense *dn, const double *d_x, const double *d_xs, const double *d_bd,
                             const double *d_f, const double *d_t, const double *d_link, double eta, double *d_res_fib,
                             double *d_out_shell, double *d_v_bodies) {
    const long long n_fw = fl->fb - fl->fa, n_sw = fl->sb - fl->sa, n_bw = fl->bb - fl->ba;
    SKB_TRY(fl->in_fib.ensure((size_t)n_fw * 24 + 8));
    SKB_TRY(fl->vel.ensure((size_t)fl->n_win * 24 + 8));
    // res_shell's dense part, stresslet_plus_complementary_ * x_shell (system.cpp:319, periphery.cpp:38-47), depends on
    // x_shell only: it is handed to the background streamer, which matvec_core launches as soon as x_shell is complete
    // on this device -- the caller's vector without a group, the gathered copy in the window with one
    skb_flow::Overlap &B = fl->bg;
    B.dn = nullptr;
    B.launched = false;
    const bool dense_rows = dn && n_sw > 0 && d_out_shell;
    if (dense_rows && B.enabled) {
        SKB_TRY(overlap_buffers(fl, 3 * n_sw));
        B.dn = dn;
        B.d_x = fl->grp.size > 1 ? fl->grp.at<double>(fl->grp.rank, fl->grp.off_xshell[(fl->grp.epoch + 1) & 1]) : d_xs;
    }
    // MatrixXd fw = fc.apply_fiber_force(x_fibers)                       system.cpp:298
    SKB_TRY(fiber_force_dev(fl, d_x, (double *)fl->in_fib.ptr));
    // v_all of system.cpp:299-316 (own rows)
    SKB_TRY(matvec_core(fl, (const double *)fl->in_fib.ptr, d_xs, d_bd, d_f, d_t, eta, (double *)fl->vel.ptr));
    // res_fibers = fc.matvec(x_fibers, v_fibers, fiber_link_conditions)   system.cpp:318
    SKB_TRY(fiber_matvec_dev(fl, d_x, (const double *)fl->vel.ptr, d_link, d_res_fib));
    const double *d_v_shell = (const double *)fl->vel.ptr + 3 * n_fw;
    if (n_sw > 0 && d_out_shell) {
        if (dense_rows && B.launched) {
            // res_shell = A x (background) + v_shell
            CUDA_TRY(cudaStreamWaitEvent(fl->cur, B.join, 0));
            add_out_kernel<<<(unsigned)((3 * n_sw + 255) / 256), 256, 0, fl->cur>>>(d_out_shell, (const double *)B.y.ptr,
                                                                                   d_v_shell, 3 * n_sw);
            SKB_TRY(launched(fl, 1));
        } else if (dn) {
            // res_shell = shell.matvec(x_shell, v_shell) = stresslet_plus_complementary_ * x_shell + v_shell in one
            // kernel at the end of the stream (skb_flow_set_overlap(fl, 0))
            const double *d_x_full = d_xs;
            if (fl->grp.size > 1)
                d_x_full = fl->grp.at<double>(fl->grp.rank, fl->grp.off_xshell[fl->grp.epoch & 1]);
            SKB_TRY(skb_dense_apply_device(dn, SKB_DENSE_STRESSLET_PLUS_COMPLEMENTARY, d_x_full, d_v_shell, d_out_shell,
                                           fl->cur));
            fl->launches += 1;
        } else {
            CUDA_TRY(cudaMemcpyAsync(d_out_shell, d_v_shell, (size_t)n_sw * 24, cudaMemcpyDeviceToDevice, fl->cur));
        }
    }
    B.dn = nullptr;
    if (n_bw > 0 && d_v_bodies)
        CUDA_TRY(cudaMemcpyAsync(d_v_bodies, (const double *)fl->vel.ptr + 3 * (n_fw + n_sw), (size_t)n_bw * 24,
                                 cudaMemcpyDeviceToDevice, fl->cur));
    return SKB_OK;
}

static int check_dense_handle(skb_flow *fl, skb_dense *dn, const char *who) {
    int dn_dev = -1;
    SKB_TRY(skb_dense_device(dn, 0, &dn_dev));
    if (fl->dev != dn_dev)
        return set_error(SKB_ERR_INVALID, "%s: the flow is on device %d, the dense handle on device %d", who, fl->dev,
                         dn_dev);
    SKB_TRY(prepare_matvec_targets(fl));
    int64_t rows = 0, cols = 0;
    SKB_TRY(skb_dense_shape(dn, SKB_DENSE_STRESSLET_PLUS_COMPLEMENTARY, &rows, &cols));
    const long long want_rows = 3 * (fl->sb - fl->sa);
    if (rows != want_rows || cols != 3 * fl->n_shell)
        return set_error(SKB_ERR_INVALID, "%s: stresslet_plus_complementary is %lld x %lld, need the %lld own rows x %lld",
                         who, (long long)rows, (long long)cols, want_rows, 3 * fl->n_shell);
    return SKB_OK;
}

// shared body of skb_flow_apply_matvec / skb_flow_apply_matvec_dense; dn != NULL: out_shell = res_shell
static int apply_matvec_impl(skb_flow *fl, skb_dense *dn, const double *x_fibers, const double *shell_density,
                             const double *body_densities, const double *body_forces_torques,
                             const double *fiber_link_conditions, double eta, double *res_fibers, double *v_shell,
                             double *v_bodies) {
    if (!fl || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_matvec: bad arguments");
    SKB_TRY(need_ops(fl, "skb_flow_apply_matvec"));
    const long long nf = fl->n_fib, ns = fl->n_shell, nb = fl->n_body, n_all = nf + ns + nb;
    if ((nf > 0 && (!x_fibers || !res_fibers)) || (ns > 0 && (!shell_density || !v_shell)) ||
        (nb > 0 && (!body_densities || !v_bodies)) || (fl->n_bodies > 0 && !body_forces_torques))
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_matvec: NULL argument for a non-empty class");
    SKB_TRY(begin_call(fl));
    if (n_all == 0)
        return SKB_OK;
    SKB_TRY(prepare_matvec_targets(fl));
    if (fl->n_win != n_all || fl->grp.size > 1)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_matvec needs the full target window (have %lld of %lld "
                                          "rows); group members use skb_flow_apply_matvec_device / skb_mflow_*",
                         fl->n_win, n_all);
    std::vector<double> f, t;
    if (fl->n_bodies > 0)
        split_forces_torques(body_forces_torques, fl->n_bodies, f, t);
    SKB_TRY(host_call_start(fl));
    if (nf)
        CUDA_TRY(cudaMemcpyAsync(fl->x_fib.ptr, x_fibers, (size_t)nf * 32, cudaMemcpyHostToDevice, fl->stream));
    if (nf && fiber_link_conditions)
        CUDA_TRY(cudaMemcpyAsync(fl->vb.ptr, fiber_link_conditions, (size_t)(fl->op_f1 - fl->op_f0) * 56,
                                 cudaMemcpyHostToDevice, fl->stream));
    SKB_TRY(upload(fl, fl->in_shell, shell_density, (size_t)ns * 3));
    SKB_TRY(upload(fl, fl->in_body, body_densities, (size_t)nb * 3));
    SKB_TRY(upload(fl, fl->in_force, f.data(), f.size()));
    SKB_TRY(upload(fl, fl->in_torque, t.data(), t.size()));
    SKB_TRY(fl->res_shell.ensure((size_t)ns * 24 + 8));
    SKB_TRY(fl->tmp_b.ensure((size_t)nb * 24 + 8));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(apply_matvec_core(fl, dn, (const double *)fl->x_fib.ptr, (const double *)fl->in_shell.ptr,
                              (const double *)fl->in_body.ptr, (const double *)fl->in_force.ptr,
                              (const double *)fl->in_torque.ptr,
                              (nf && fiber_link_conditions) ? (const double *)fl->vb.ptr : nullptr, eta,
                              (double *)fl->res_fib.ptr, (double *)fl->res_shell.ptr, (double *)fl->tmp_b.ptr));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    if (nf)
        CUDA_TRY(cudaMemcpyAsync(res_fibers, fl->res_fib.ptr, (size_t)nf * 32, cudaMemcpyDeviceToHost, fl->stream));
    if (ns)
        CUDA_TRY(cudaMemcpyAsync(v_shell, fl->res_shell.ptr, (size_t)ns * 24, cudaMemcpyDeviceToHost, fl->stream));
    if (nb)
        CUDA_TRY(cudaMemcpyAsync(v_bodies, fl->tmp_b.ptr, (size_t)nb * 24, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl);
}

// =====================================================================================================================
// skb_mflow -- ONE process, n GPUs (include/skelly_b200_flow.h): the multi-device shape the reference's "direct
// evaluators need a single rank" rule admits (src/core/system.cpp:618-623).  One group member (skb_flow) per device,
// connected through peer memory; whole fibers, periphery rows and body rows are block-partitioned over the members.
// Every member is driven by its own host thread, so the n launch sequences are issued concurrently.
// =====================================================================================================================
namespace {
class Workers {
  public:
    explicit Workers(int n) : n_(n), task_(n), state_(n, 0), rc_(n, 0), msg_(n) {
        for (int g = 0; g < n; ++g)
            th_.emplace_back([this, g] { loop(g); });
    }
    ~Workers() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : th_)
            t.join();
    }
    // run fn(g) on every worker; returns the first non-zero status (its message becomes this thread's last error)
    int run(const std::function<int(int)> &fn) {
        {
            std::lock_guard<std::mutex> lk(mu_);
            for (int g = 0; g < n_; ++g) {
                task_[g] = fn;
                state_[g] = 1;
            }
        }
        cv_.notify_all();
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [this] {
            for (int g = 0; g < n_; ++g)
                if (state_[g] != 0)
                    return false;
            return true;
        });
        for (int g = 0; g < n_; ++g)
            if (rc_[g] != SKB_OK)
                return set_error(rc_[g], "device member %d: %s", g, msg_[g].c_str());
        return SKB_OK;
    }

  private:
    void loop(int g) {
        for (;;) {
            std::function<int(int)> fn;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this, g] { return stop_ || state_[g] == 1; });
                if (stop_)
                    return;
                fn = task_[g];
            }
            const int rc = fn(g);
            {
                std::lock_guard<std::mutex> lk(mu_);
                rc_[g] = rc;
                msg_[g] = rc == SKB_OK ? "" : last_error();
                state_[g] = 0;
            }
            done_.notify_all();
        }
    }
    int n_;
    std::vector<std::function<int(int)>> task_;
    std::vector<int> state_, rc_;
    std::vector<std::string> msg_;
    std::vector<std::thread> th_;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    bool stop_ = false;
};
} // namespace

struct skb_mflow {
    int n = 0;
    std::vector<int> devs;
    std::vector<skb_flow *> m;
    std::vector<skb_dense *> dn;
    std::unique_ptr<Workers> workers;
    // geometry (host copies of what the partition needs)
    long long n_fib = 0, n_shell = 0, n_body = 0;
    int n_fibers = 0, n_bodies = 0;
    std::vector<int> fiber_n;
    std::vector<long long> fiber_off;
    // partition: member g owns fibers [f0[g], f1[g]), periphery rows [s0, s1), body rows [b0, b1)
    std::vector<int> f0, f1;
    std::vector<long long> s0, s1, b0, b1;
    bool part_dirty = true;
    bool has_dense = false;
    bool ops_ready = false;
    struct IO { // per-member device buffers of the host-pointer calls
        DevBuf x, xs, bd, f, t, link, res, outs, vb, ff, v;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
    };
    std::vector<IO> io;
    skb_flow_stats stats{};
};

// member g of n owns whole fibers [f0, f1) -- cut where the running node count passes g/n of the total
// (fcfd.cpp:102-120 splits by fiber count; by node count balances ragged suspensions as well) -- and equal blocks of
// the periphery and body rows
static void partition_rows(const std::vector<long long> &fiber_off, long long n_shell, long long n_body, int n,
                           std::vector<int> &f0, std::vector<int> &f1, std::vector<long long> &s0,
                           std::vector<long long> &s1, std::vector<long long> &b0, std::vector<long long> &b1) {
    const int n_fibers = (int)fiber_off.size() - 1;
    const long long n_fib = n_fibers > 0 ? fiber_off[(size_t)n_fibers] : 0;
    f0.assign(n, 0), f1.assign(n, 0);
    s0.assign(n, 0), s1.assign(n, 0), b0.assign(n, 0), b1.assign(n, 0);
    int f = 0;
    for (int g = 0; g < n; ++g) {
        f0[g] = f;
        const long long want = n_fib * (g + 1) / n;
        while (f < n_fibers && fiber_off[(size_t)f + 1] <= want)
            ++f;
        if (g == n - 1)
            f = std::max(n_fibers, 0);
        f1[g] = f;
    }
    const long long cs = (n_shell + n - 1) / n, cb = (n_body + n - 1) / n;
    for (int g = 0; g < n; ++g) {
        s0[g] = std::min(n_shell, g * cs);
        s1[g] = std::min(n_shell, (g + 1) * cs);
        b0[g] = std::min(n_body, g * cb);
        b1[g] = std::min(n_body, (g + 1) * cb);
    }
}

static void mflow_partition(skb_mflow *mf) {
    std::vector<long long> off = mf->fiber_off;
    if (off.empty())
        off.push_back(0);
    partition_rows(off, mf->n_shell, mf->n_body, mf->n, mf->f0, mf->f1, mf->s0, mf->s1, mf->b0, mf->b1);
}

// ranges + group wiring, after any change of the geometry's sizes
static int mflow_prepare(skb_mflow *mf) {
    if (!mf->part_dirty)
        return SKB_OK;
    mflow_partition(mf);
    for (int g = 0; g < mf->n; ++g) {
        SKB_TRY(skb_flow_set_target_ranges(mf->m[g], mf->f0[g], mf->f1[g], mf->s0[g], mf->s1[g], mf->b0[g], mf->b1[g]));
        SKB_TRY(skb_flow_group_init(mf->m[g], g, mf->n));
    }
    for (int g = 0; g < mf->n; ++g)
        for (int h = 0; h < mf->n; ++h)
            if (g != h)
                SKB_TRY(skb_flow_group_connect(mf->m[g], h, mf->m[h]));
    for (int g = 0; g < mf->n; ++g) // all allocations up front: members may share a device (see skb_flow_group_warmup)
        SKB_TRY(skb_flow_group_warmup(mf->m[g]));
    mf->part_dirty = false;
    mf->ops_ready = false;
    return SKB_OK;
}

// element offset of fiber f's block in a concatenation of per-fiber (k n) x (4 n) matrices
static long long op_offset(const skb_mflow *mf, int f, int k) {
    long long o = 0;
    for (int i = 0; i < f; ++i)
        o += (long long)k * 4 * mf->fiber_n[(size_t)i] * mf->fiber_n[(size_t)i];
    return o;
}

// the members' last stats summed; device_ms = total_ms = the slowest member's device_ms
static void mflow_sum_stats(skb_mflow *mf) {
    skb_flow_stats sum{};
    for (int g = 0; g < mf->n; ++g) {
        skb_flow_stats st{};
        skb_flow_last_stats(mf->m[g], &st);
        sum.device_ms = std::max(sum.device_ms, st.device_ms);
        sum.n_pairs += st.n_pairs;
        sum.launches += st.launches;
    }
    sum.total_ms = sum.device_ms;
    mf->stats = sum;
}

// after a group call: the members' stats summed, each member timed by its io events (its device calls take no times)
static int mflow_collect_stats(skb_mflow *mf) {
    double dev_ms = 0;
    for (int g = 0; g < mf->n; ++g) {
        float ms = 0;
        cudaSetDevice(mf->devs[g]);
        if (cudaEventElapsedTime(&ms, mf->io[g].e0, mf->io[g].e1) == cudaSuccess)
            dev_ms = std::max(dev_ms, (double)ms);
        else
            (void)cudaGetLastError();
        int missing = -1;
        SKB_TRY(skb_flow_group_error(mf->m[g], &missing));
        if (missing >= 0)
            return set_error(SKB_ERR_STATE, "device member %d timed out waiting for member %d (a peer failed or never "
                                            "issued the matching call)", g, missing);
    }
    mflow_sum_stats(mf);
    mf->stats.device_ms = mf->stats.total_ms = dev_ms;
    return SKB_OK;
}

// member g's rows: its first fiber node a, its fiber nodes, periphery rows and body rows
struct MemberRows {
    long long a, n_fw, n_sw, n_bw;
};
static MemberRows member_rows(const skb_mflow *mf, int g) {
    const long long a = mf->fiber_off.empty() ? 0 : mf->fiber_off[(size_t)mf->f0[g]],
                    b = mf->fiber_off.empty() ? 0 : mf->fiber_off[(size_t)mf->f1[g]];
    return MemberRows{a, b - a, mf->s1[g] - mf->s0[g], mf->b1[g] - mf->b0[g]};
}

// Size every member's transfer buffers on the CALLING thread, before any member starts launching: cudaMalloc /
// cudaFree may synchronise the whole device and must not run while a peer on the same device sits in a flag wait.
static int mflow_size_io(skb_mflow *mf, size_t n_ft) {
    for (int g = 0; g < mf->n; ++g) {
        CUDA_TRY(cudaSetDevice(mf->devs[g]));
        skb_mflow::IO &io = mf->io[g];
        const MemberRows r = member_rows(mf, g);
        const size_t n_fw = (size_t)r.n_fw, n_sw = (size_t)r.n_sw, n_bw = (size_t)r.n_bw;
        const size_t n_fibers = (size_t)(mf->f1[g] - mf->f0[g]);
        SKB_TRY(io.x.ensure(n_fw * 32 + 8));
        SKB_TRY(io.ff.ensure(n_fw * 24 + 8));
        SKB_TRY(io.xs.ensure(n_sw * 24 + 8));
        SKB_TRY(io.bd.ensure((size_t)mf->n_body * 24 + 8));
        SKB_TRY(io.f.ensure(n_ft * 8 + 8));
        SKB_TRY(io.t.ensure(n_ft * 8 + 8));
        SKB_TRY(io.link.ensure(n_fibers * 56 + 8));
        SKB_TRY(io.res.ensure(n_fw * 32 + 8));
        SKB_TRY(io.outs.ensure(n_sw * 24 + 8));
        SKB_TRY(io.vb.ensure(n_bw * 24 + 8));
        SKB_TRY(io.v.ensure((n_fw + n_sw + n_bw) * 24 + 8));
        if (mf->has_dense && n_sw > 0 && mf->m[g]->bg.enabled)
            SKB_TRY(overlap_buffers(mf->m[g], 3 * (long long)n_sw));
    }
    return SKB_OK;
}

extern "C" {

int skb_flow_create(int device, skb_flow **out) {
    if (!out)
        return set_error(SKB_ERR_INVALID, "skb_flow_create: out == NULL");
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
        return set_error(SKB_ERR_NO_DEVICE, "no CUDA device available; this library has no CPU fallback");
    if (device < 0 || device >= n_dev)
        return set_error(SKB_ERR_INVALID, "skb_flow_create: device %d out of range (%d visible)", device, n_dev);
    std::unique_ptr<skb_flow> fl(new skb_flow);
    fl->dev = device;
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaStreamCreateWithFlags(&fl->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&fl->ev0));
    CUDA_TRY(cudaEventCreate(&fl->ev1));
    CUDA_TRY(cudaEventCreate(&fl->evt0));
    CUDA_TRY(cudaEventCreate(&fl->evt1));
    if (const char *e = getenv("SKB_GRAPHS"))
        fl->graphs_enabled = atoi(e) != 0;
    if (const char *e = getenv("SKB_OVERLAP")) // A/B switch of skb_flow_set_overlap's default
        fl->bg.enabled = atoi(e) != 0;
    for (int k = 0; k < 2; ++k) {
        SKB_TRY(ensure_ctx(fl.get(), &fl->fib[k]));
        SKB_TRY(ensure_ctx(fl.get(), &fl->shell[k]));
        SKB_TRY(ensure_ctx(fl.get(), &fl->body[k]));
    }
    // empty classes until set_* is called
    for (int k = 0; k < 2; ++k) {
        SKB_TRY(skb_set_sources(fl->fib[k], SKB_STOKESLET, nullptr, 0));
        SKB_TRY(skb_set_sources(fl->shell[k], SKB_STRESSLET, nullptr, 0));
        SKB_TRY(skb_set_sources(fl->body[k], SKB_STRESSLET, nullptr, 0));
        SKB_TRY(skb_set_sources(fl->body[k], SKB_STOKESLET, nullptr, 0));
    }
    *out = fl.release();
    return SKB_OK;
}

int skb_flow_destroy(skb_flow *fl) {
    if (!fl)
        return SKB_OK;
    cudaSetDevice(fl->dev);
    if (fl->stream)
        cudaStreamSynchronize(fl->stream);
    for (int k = 0; k < 2; ++k) {
        skb_ctx_destroy(fl->fib[k]);
        skb_ctx_destroy(fl->shell[k]);
        skb_ctx_destroy(fl->body[k]);
    }
    DevBuf *bufs[] = {&fl->fiber_offset, &fl->fiber_length, &fl->r_fib, &fl->r_shell, &fl->r_body, &fl->centers,
                      &fl->pt_pos, &fl->pt_force, &fl->pt_torque, &fl->in_fib, &fl->in_shell, &fl->in_body, &fl->in_force, &fl->in_torque, &fl->vel, &fl->tmp,
                      &fl->op_A, &fl->op_F, &fl->op_xs, &fl->op_len, &fl->op_plus, &fl->op_class, &fl->op_classD,
                      &fl->op_classP, &fl->op_classR, &fl->op_ranges, &fl->items_A, &fl->items_F, &fl->x_fib, &fl->res_fib, &fl->vb, &fl->res_shell, &fl->op_Ainv, &fl->tmp_b};
    for (DevBuf *b : bufs)
        b->release();
    fl->g_matvec.reset();
    fl->g_vat.reset();
    group_release(fl);
    fl->scratch_u.release();
    fl->cross.release();
    fl->bg.y.release();
    if (fl->bg.fork) cudaEventDestroy(fl->bg.fork);
    if (fl->bg.join) cudaEventDestroy(fl->bg.join);
    if (fl->bg.stream) cudaStreamDestroy(fl->bg.stream);
    if (fl->h_stage)
        cudaFreeHost(fl->h_stage);
    if (fl->ev0) cudaEventDestroy(fl->ev0);
    if (fl->ev1) cudaEventDestroy(fl->ev1);
    if (fl->evt0) cudaEventDestroy(fl->evt0);
    if (fl->evt1) cudaEventDestroy(fl->evt1);
    if (fl->stream) cudaStreamDestroy(fl->stream);
    delete fl;
    return SKB_OK;
}

int skb_flow_set_fibers(skb_flow *fl, const double *r_fib, const int *n_nodes, const double *length, int n_fibers) {
    if (!fl || n_fibers < 0 || (n_fibers > 0 && (!r_fib || !n_nodes || !length)))
        return set_error(SKB_ERR_INVALID, "skb_flow_set_fibers: bad arguments");
    std::vector<long long> off((size_t)n_fibers + 1, 0);
    int max_n = 0;
    for (int f = 0; f < n_fibers; ++f) {
        if (n_nodes[f] < 2)
            return set_error(SKB_ERR_INVALID, "fiber %d has %d nodes (need >= 2)", f, n_nodes[f]);
        off[f + 1] = off[f] + n_nodes[f];
        max_n = std::max(max_n, n_nodes[f]);
    }
    if ((size_t)max_n * 48 > 200 * 1024)
        return set_error(SKB_ERR_INVALID, "fiber with %d nodes exceeds the shared-memory self-term kernel", max_n);
    fl->n_fibers = n_fibers;
    fl->n_fib = off[n_fibers];
    fl->max_fiber_nodes = max_n;
    fl->h_r_fib.assign(r_fib, r_fib + 3 * fl->n_fib);
    fl->h_fiber_n.assign(n_nodes, n_nodes + n_fibers);
    fl->h_fiber_off = off;
    fl->ops_ready = false; // operators belong to one set of fibers
    fl->mv_dirty = true;
    fl->geom_version++;
    CUDA_TRY(cudaSetDevice(fl->dev));
    for (int k = 0; k < 2; ++k)
        SKB_TRY(skb_set_sources(fl->fib[k], SKB_STOKESLET, r_fib, fl->n_fib));
    if (n_fibers == 0)
        return SKB_OK;
    SKB_TRY(fl->fiber_offset.ensure(off.size() * 8));
    SKB_TRY(fl->fiber_length.ensure((size_t)n_fibers * 8));
    SKB_TRY(fl->r_fib.ensure((size_t)fl->n_fib * 24));
    CUDA_TRY(cudaMemcpyAsync(fl->fiber_offset.ptr, off.data(), off.size() * 8, cudaMemcpyHostToDevice, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(fl->fiber_length.ptr, length, (size_t)n_fibers * 8, cudaMemcpyHostToDevice, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(fl->r_fib.ptr, r_fib, (size_t)fl->n_fib * 24, cudaMemcpyHostToDevice, fl->stream));
    if (max_n * 48 > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(fiber_self_subtract_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      max_n * 48));
    // trapezoid weights straight into both Stokeslet source sets
    for (int k = 0; k < 2; ++k) {
        SourceSet &s = fl->fib[k]->devs[0].src[SKB_STOKESLET];
        SKB_TRY(s.weights.ensure((size_t)fl->n_fib * 8));
        fiber_weights_kernel<<<n_fibers, 64, 0, fl->stream>>>((const long long *)fl->fiber_offset.ptr,
                                                              (const double *)fl->fiber_length.ptr, n_fibers,
                                                              (double *)s.weights.ptr);
        SKB_TRY(launched(fl, 1));
        s.has_weights = true;
    }
    CUDA_TRY(cudaStreamSynchronize(fl->stream));
    return SKB_OK;
}

int skb_flow_set_periphery(skb_flow *fl, const double *node_pos, const double *node_normal, int64_t n_nodes) {
    if (!fl || n_nodes < 0 || (n_nodes > 0 && (!node_pos || !node_normal)))
        return set_error(SKB_ERR_INVALID, "skb_flow_set_periphery: bad arguments");
    fl->n_shell = n_nodes;
    fl->h_r_shell.assign(node_pos, node_pos + 3 * n_nodes);
    fl->mv_dirty = true;
    fl->geom_version++;
    for (int k = 0; k < 2; ++k) {
        SKB_TRY(skb_set_sources(fl->shell[k], SKB_STRESSLET, node_pos, n_nodes));
        SKB_TRY(skb_set_source_normals(fl->shell[k], node_normal, n_nodes));
    }
    return SKB_OK;
}

int skb_flow_set_bodies(skb_flow *fl, const double *node_pos, const double *node_normal, int64_t n_nodes,
                        const double *centers, int n_bodies) {
    if (!fl || n_nodes < 0 || n_bodies < 0 || (n_nodes > 0 && (!node_pos || !node_normal)) ||
        (n_bodies > 0 && !centers) || (n_bodies == 0 && n_nodes > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_set_bodies: bad arguments");
    fl->n_body = n_nodes;
    fl->n_bodies = n_bodies;
    fl->h_r_body.assign(node_pos, node_pos + 3 * n_nodes);
    fl->mv_dirty = true;
    fl->geom_version++;
    for (int k = 0; k < 2; ++k) {
        SKB_TRY(skb_set_sources(fl->body[k], SKB_STRESSLET, node_pos, n_nodes));
        SKB_TRY(skb_set_source_normals(fl->body[k], node_normal, n_nodes));
        SKB_TRY(skb_set_sources(fl->body[k], SKB_STOKESLET, centers, n_bodies));
    }
    if (n_bodies > 0) {
        CUDA_TRY(cudaSetDevice(fl->dev));
        SKB_TRY(fl->centers.ensure((size_t)n_bodies * 24));
        CUDA_TRY(cudaMemcpyAsync(fl->centers.ptr, centers, (size_t)n_bodies * 24, cudaMemcpyHostToDevice, fl->stream));
        CUDA_TRY(cudaStreamSynchronize(fl->stream));
    }
    return SKB_OK;
}

int skb_flow_fibers(skb_flow *fl, const double *r_trg, int64_t n_trg, const double *fib_forces, double eta,
                    int subtract_self, double *vel) {
    if (!fl || n_trg < 0 || (n_trg > 0 && (!r_trg || !vel)) || (fl->n_fib > 0 && !fib_forces) || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_fibers: bad arguments");
    SKB_TRY(begin_call(fl));
    SKB_TRY(set_targets_cached(fl->fib[0], fl->tc_fib, r_trg, n_trg));
    if (n_trg == 0)
        return SKB_OK;
    SKB_TRY(host_call_start(fl));
    SKB_TRY(upload(fl, fl->in_fib, fib_forces, (size_t)fl->n_fib * 3));
    SKB_TRY(fl->vel.ensure((size_t)n_trg * 24));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(fibers_dev(fl, fl->fib[0], (const double *)fl->in_fib.ptr, eta, subtract_self, (double *)fl->vel.ptr, 0, 0,
                       fl->n_fib));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(vel, fl->vel.ptr, (size_t)n_trg * 24, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl);
}

int skb_flow_periphery(skb_flow *fl, const double *r_trg, int64_t n_trg, const double *density, double eta,
                       double *vel) {
    if (!fl || n_trg < 0 || (n_trg > 0 && (!r_trg || !vel)) || (fl->n_shell > 0 && !density) || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_periphery: bad arguments");
    SKB_TRY(begin_call(fl));
    SKB_TRY(set_targets_cached(fl->shell[0], fl->tc_shell, r_trg, n_trg));
    if (n_trg == 0)
        return SKB_OK;
    SKB_TRY(host_call_start(fl));
    SKB_TRY(upload(fl, fl->in_shell, density, (size_t)fl->n_shell * 3));
    SKB_TRY(fl->vel.ensure((size_t)n_trg * 24));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(periphery_dev(fl, fl->shell[0], kNormalDensity, (const double *)fl->in_shell.ptr, eta,
                          (double *)fl->vel.ptr, 0));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(vel, fl->vel.ptr, (size_t)n_trg * 24, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl);
}

int skb_flow_bodies(skb_flow *fl, const double *r_trg, int64_t n_trg, const double *densities,
                    const double *forces_torques, double eta, double *vel) {
    if (!fl || n_trg < 0 || (n_trg > 0 && (!r_trg || !vel)) || (fl->n_body > 0 && !densities) ||
        (fl->n_bodies > 0 && !forces_torques) || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_bodies: bad arguments");
    SKB_TRY(begin_call(fl));
    SKB_TRY(set_targets_cached(fl->body[0], fl->tc_body, r_trg, n_trg));
    if (n_trg == 0)
        return SKB_OK;
    std::vector<double> f, t;
    split_forces_torques(forces_torques, fl->n_bodies, f, t);
    SKB_TRY(host_call_start(fl));
    SKB_TRY(upload(fl, fl->in_body, densities, (size_t)fl->n_body * 3));
    SKB_TRY(upload(fl, fl->in_force, f.data(), f.size()));
    SKB_TRY(upload(fl, fl->in_torque, t.data(), t.size()));
    SKB_TRY(fl->vel.ensure((size_t)n_trg * 24));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(bodies_dev(fl, fl->body[0], (const double *)fl->in_body.ptr, (const double *)fl->in_force.ptr,
                       (const double *)fl->in_torque.ptr, eta, (double *)fl->vel.ptr, 0));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(vel, fl->vel.ptr, (size_t)n_trg * 24, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl); // (it waits for the stream: f, t are stack-owned staging)
}

int skb_flow_set_point_sources(skb_flow *fl, const double *positions, const double *forces, const double *torques,
                               int n_points) {
    if (!fl || n_points < 0 || (n_points > 0 && (!positions || !forces || !torques)))
        return set_error(SKB_ERR_INVALID, "skb_flow_set_point_sources: bad arguments");
    fl->n_points = n_points;
    fl->geom_version++;
    if (n_points == 0)
        return SKB_OK;
    CUDA_TRY(cudaSetDevice(fl->dev));
    SKB_TRY(fl->pt_pos.ensure((size_t)n_points * 24));
    SKB_TRY(fl->pt_force.ensure((size_t)n_points * 24));
    SKB_TRY(fl->pt_torque.ensure((size_t)n_points * 24));
    CUDA_TRY(cudaMemcpyAsync(fl->pt_pos.ptr, positions, (size_t)n_points * 24, cudaMemcpyHostToDevice, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(fl->pt_force.ptr, forces, (size_t)n_points * 24, cudaMemcpyHostToDevice, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(fl->pt_torque.ptr, torques, (size_t)n_points * 24, cudaMemcpyHostToDevice, fl->stream));
    CUDA_TRY(cudaStreamSynchronize(fl->stream));
    return SKB_OK;
}

int skb_flow_set_background(skb_flow *fl, const int *components, const double *scale_factor, const double *uniform) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_background: NULL");
    fl->geom_version++;
    if (!components || !scale_factor || !uniform) {
        fl->has_background = false;
        return SKB_OK;
    }
    for (int j = 0; j < 3; ++j) {
        if (components[j] < 0 || components[j] > 2)
            return set_error(SKB_ERR_INVALID, "skb_flow_set_background: components must be 0, 1 or 2");
        fl->bg_comp[j] = components[j];
        fl->bg_scale[j] = scale_factor[j];
        fl->bg_uniform[j] = uniform[j];
    }
    fl->has_background = true;
    return SKB_OK;
}

int skb_flow_velocity_at_targets(skb_flow *fl, const double *r_trg, int64_t n_trg, const double *fib_forces,
                                 const double *shell_density, const double *body_densities,
                                 const double *body_forces_torques, double eta, double *vel) {
    if (!fl || n_trg < 0 || (n_trg > 0 && (!r_trg || !vel)) || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_velocity_at_targets: bad arguments");
    if ((fl->n_fib > 0 && !fib_forces) || (fl->n_shell > 0 && !shell_density) || (fl->n_body > 0 && !body_densities) ||
        (fl->n_bodies > 0 && !body_forces_torques))
        return set_error(SKB_ERR_INVALID, "skb_flow_velocity_at_targets: NULL input for a non-empty class");
    SKB_TRY(begin_call(fl));
    // the three "arbitrary target" evaluators share one cached target list
    SKB_TRY(set_targets_cached(fl->fib[0], fl->tc_fib, r_trg, n_trg));
    SKB_TRY(set_targets_cached(fl->shell[0], fl->tc_shell, r_trg, n_trg));
    SKB_TRY(set_targets_cached(fl->body[0], fl->tc_body, r_trg, n_trg));
    if (n_trg == 0)
        return SKB_OK;
    std::vector<double> f, t;
    if (fl->n_bodies > 0)
        split_forces_torques(body_forces_torques, fl->n_bodies, f, t);
    SKB_TRY(fl->vel.ensure((size_t)n_trg * 24));
    double *d_v = (double *)fl->vel.ptr;
    // device-side sequence with the strengths at `in` and the velocities going to v_host
    auto body = [&](const HostStrengths &in, double *v_host) -> int {
        SKB_TRY(upload_strengths(fl, in));
        // fc_->flow(r_trg, f_on_fibers, eta, /*subtract_self=*/false) + bc_.flow + shell_->flow   system.cpp:355-359
        SKB_TRY(fibers_dev(fl, fl->fib[0], (const double *)fl->in_fib.ptr, eta, 0, d_v, 0, 0, 0));
        SKB_TRY(bodies_dev(fl, fl->body[0], (const double *)fl->in_body.ptr, (const double *)fl->in_force.ptr,
                           (const double *)fl->in_torque.ptr, eta, d_v, 1));
        SKB_TRY(periphery_dev(fl, fl->shell[0], kNormalDensity, (const double *)fl->in_shell.ptr, eta, d_v, 1));
        // + psc_.flow(r_trg, eta, time) + bs_.flow(r_trg, eta)                                  system.cpp:358-359
        const double *d_trg = (const double *)fl->fib[0]->devs[0].r_trg.ptr;
        const int bs = 128;
        const unsigned nblk = (unsigned)((n_trg + bs - 1) / bs);
        if (fl->n_points > 0) {
            oseen_contract_add_kernel<<<nblk, bs, 0, fl->stream>>>((const double *)fl->pt_pos.ptr,
                                                                   (const double *)fl->pt_force.ptr, fl->n_points,
                                                                   d_trg, n_trg, 1.0 / (8.0 * M_PI * eta),
                                                                   kReg * kReg, kEps, d_v);
            rotlet_add_kernel<<<nblk, bs, 0, fl->stream>>>((const double *)fl->pt_pos.ptr,
                                                           (const double *)fl->pt_torque.ptr, fl->n_points, d_trg,
                                                           n_trg, 1.0 / (8.0 * M_PI * eta), kReg * kReg, kEps * kEps,
                                                           d_v);
            SKB_TRY(launched(fl, 2));
        }
        if (fl->has_background) {
            background_add_kernel<<<nblk, bs, 0, fl->stream>>>(d_trg, n_trg, fl->bg_comp[0], fl->bg_comp[1],
                                                               fl->bg_comp[2], fl->bg_scale[0], fl->bg_scale[1],
                                                               fl->bg_scale[2], fl->bg_uniform[0], fl->bg_uniform[1],
                                                               fl->bg_uniform[2], d_v);
            SKB_TRY(launched(fl, 1));
        }
        CUDA_TRY(cudaMemcpyAsync(v_host, d_v, (size_t)n_trg * 24, cudaMemcpyDeviceToHost, fl->stream));
        return SKB_OK;
    };
    const HostStrengths in{fib_forces, shell_density, body_densities, f.data(), t.data()};
    const size_t n_out = (size_t)n_trg * 3;
    SKB_TRY(host_call_start(fl));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    // the listener / streamline integrator asks for 1-6 targets per call (streamline.cpp:11-35): launch-bound
    const bool graphed = fl->graphs_enabled && (n_strengths(fl) + n_out) * 8 <= kGraphMaxBytes;
    double *h_v = nullptr;
    if (graphed) {
        HostStrengths staged;
        SKB_TRY(fill_stage(fl, in, n_out, &staged, &h_v));
        unsigned long long key = mix_key(fl->geom_version, (unsigned long long)n_trg);
        key = mix_key(key, dbl_bits(eta));
        key = mix_key(key, buffer_key(fl, 0));
        // same count but different targets: the captured sequence assumed the old targets' relation to the sources
        key = mix_key(key, fl->tc_fib.version);
        key = mix_key(key, fl->tc_shell.version);
        key = mix_key(key, fl->tc_body.version);
        SKB_TRY(run_graphed(fl, fl->g_vat, key, [&]() { return body(staged, h_v); }));
    } else {
        SKB_TRY(body(in, vel));
    }
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    SKB_TRY(host_call_finish(fl));
    if (graphed)
        std::memcpy(vel, h_v, n_out * 8);
    return SKB_OK;
}

// ---- group membership (multi-GPU through peer memory, group_kernels.cuh) -----------------------------------------

int skb_flow_group_init(skb_flow *fl, int rank, int size) {
    if (!fl || size < 1 || size > kMaxGroup || rank < 0 || rank >= size)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_init: need 0 <= rank < size <= %d", kMaxGroup);
    CUDA_TRY(cudaSetDevice(fl->dev));
    CUDA_TRY(cudaStreamSynchronize(fl->stream));
    group_release(fl);
    fl->mv_dirty = true;
    fl->ops_ready = false;
    fl->geom_version++;
    if (size == 1)
        return SKB_OK;
    skb_flow::Group &G = fl->grp;
    G.rank = rank;
    G.size = size;
    G.n_fib = fl->n_fib;
    G.n_shell = fl->n_shell;
    // the same padded sizes the evaluator contexts use (set_sources_impl): the window replaces their f_packed
    G.n_pad_fib = fl->n_fib > 0 ? fl->fib[1]->devs[0].src[SKB_STOKESLET].n_pad : 0;
    G.n_pad_shell = fl->n_shell > 0 ? fl->shell[1]->devs[0].src[SKB_STRESSLET].n_pad : 0;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t at = off;
        off += (bytes + 255) & ~(size_t)255;
        return at;
    };
    G.off_flags = take((size_t)(kGroupPhases * kMaxGroup + 8) * 8);
    for (int b = 0; b < 2; ++b) {
        G.off_fsl[b] = take((size_t)G.n_pad_fib * 24 + 16);
        G.off_fshell[b] = take((size_t)G.n_pad_shell * 48 + 16);
        G.off_xshell[b] = take((size_t)G.n_shell * 24 + 16);
    }
    G.off_upart = take((size_t)G.n_fib * 24 + 16);
    G.off_upart_shell = take((size_t)G.n_shell * 24 + 16);
    G.window_bytes = off;
    CUDA_TRY(cudaMalloc(&G.window, G.window_bytes));
    CUDA_TRY(cudaMemset(G.window, 0, G.window_bytes)); // flags at epoch 0, strength pads zero for good
    G.peer[rank] = G.window;
    return SKB_OK;
}

int skb_flow_group_export(skb_flow *fl, void *handle) {
    if (!fl || !handle || !fl->grp.window)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_export: no group window (skb_flow_group_init with size > 1 first)");
    static_assert(sizeof(cudaIpcMemHandle_t) == SKB_FLOW_IPC_HANDLE_BYTES, "handle size");
    CUDA_TRY(cudaSetDevice(fl->dev));
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, fl->grp.window));
    std::memcpy(handle, &h, sizeof(h));
    return SKB_OK;
}

int skb_flow_group_import(skb_flow *fl, int peer_rank, const void *handle) {
    if (!fl || !handle || !fl->grp.window || peer_rank < 0 || peer_rank >= fl->grp.size || peer_rank == fl->grp.rank)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_import: bad arguments");
    CUDA_TRY(cudaSetDevice(fl->dev));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    void *p = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    fl->grp.peer[peer_rank] = p;
    fl->grp.peer_ipc[peer_rank] = true;
    return SKB_OK;
}

int skb_flow_group_connect(skb_flow *fl, int peer_rank, skb_flow *peer) {
    if (!fl || !peer || !fl->grp.window || !peer->grp.window || peer_rank < 0 || peer_rank >= fl->grp.size ||
        peer_rank == fl->grp.rank || peer->grp.rank != peer_rank || peer->grp.size != fl->grp.size)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_connect: bad arguments");
    if (peer->grp.window_bytes != fl->grp.window_bytes || peer->grp.n_fib != fl->grp.n_fib ||
        peer->grp.n_shell != fl->grp.n_shell)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_connect: the two members were laid out for different geometries");
    CUDA_TRY(cudaSetDevice(fl->dev));
    if (peer->dev != fl->dev) {
        int can = 0;
        CUDA_TRY(cudaDeviceCanAccessPeer(&can, fl->dev, peer->dev));
        if (!can)
            return set_error(SKB_ERR_CUDA, "device %d cannot address device %d (no NVLink / P2P path)", fl->dev, peer->dev);
        cudaError_t e = cudaDeviceEnablePeerAccess(peer->dev, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled)
            (void)cudaGetLastError();
        else if (e != cudaSuccess)
            return set_error(SKB_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", fl->dev, peer->dev,
                             cudaGetErrorString(e));
    }
    fl->grp.peer[peer_rank] = peer->grp.window;
    fl->grp.peer_ipc[peer_rank] = false;
    return SKB_OK;
}

// One matvec of this member alone (no flags, own window only, zero strengths): every buffer of the path reaches its
// steady-state size, so that no cudaMalloc / cudaFree -- which synchronise the whole DEVICE -- happens later while a
// peer on the same device sits in a flag wait.  Needed when members share a GPU; harmless otherwise.
int skb_flow_group_warmup(skb_flow *fl) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_warmup: NULL flow");
    if (fl->grp.size <= 1)
        return SKB_OK;
    CUDA_TRY(cudaSetDevice(fl->dev));
    SKB_TRY(prepare_matvec_targets(fl));
    const long long n_fw = fl->fb - fl->fa, n_sw = fl->sb - fl->sa;
    DevBuf z;
    const size_t n_z = (size_t)std::max<long long>({4 * n_fw, 3 * n_sw, 3 * fl->n_body, 3LL * fl->n_bodies, 1LL});
    SKB_TRY(z.ensure(n_z * 8));
    CUDA_TRY(cudaMemsetAsync(z.ptr, 0, n_z * 8, fl->stream));
    SKB_TRY(fl->vel.ensure((size_t)fl->n_win * 24 + 8));
    SKB_TRY(fl->in_fib.ensure((size_t)n_fw * 24 + 8));
    if (n_sw > 0 && fl->bg.enabled)
        SKB_TRY(overlap_buffers(fl, 3 * n_sw));
    fl->cur = fl->stream;
    fl->grp.dry = true;
    const double *zp = (const double *)z.ptr;
    int rc = matvec_core_group(fl, zp, zp, zp, zp, zp, 1.0, (double *)fl->vel.ptr);
    fl->grp.dry = false;
    cudaError_t e = cudaStreamSynchronize(fl->stream);
    fl->grp.epoch = 0;
    z.release();
    if (rc != SKB_OK)
        return rc;
    if (e != cudaSuccess)
        return set_error(SKB_ERR_CUDA, "skb_flow_group_warmup: %s", cudaGetErrorString(e));
    return SKB_OK;
}

// Profiling aid: evaluate this member's share ALONE from now on (no flags, own window only) -- the per-rank device time
// of an n-way group on one GPU.  Results are the member's partial view, not the group's.
int skb_flow_group_set_solo(skb_flow *fl, int solo) {
    if (!fl || fl->grp.size <= 1)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_set_solo: not a group member");
    fl->grp.dry = solo != 0;
    return SKB_OK;
}

int skb_flow_group_error(skb_flow *fl, int *missing_peer) {
    if (!fl || !missing_peer)
        return set_error(SKB_ERR_INVALID, "skb_flow_group_error: NULL");
    *missing_peer = -1;
    if (!fl->grp.window)
        return SKB_OK;
    unsigned long long w = 0;
    CUDA_TRY(cudaSetDevice(fl->dev));
    CUDA_TRY(cudaMemcpy(&w, (char *)fl->grp.window + fl->grp.off_flags + (size_t)kGroupPhases * kMaxGroup * 8, 8,
                        cudaMemcpyDeviceToHost));
    if (w)
        *missing_peer = (int)(w - 1);
    return SKB_OK;
}

int skb_flow_set_cross(skb_flow *fl, int mode) {
    if (!fl || mode < -1 || mode > 1)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_cross: mode must be -1 (auto), 0 (off) or 1 (on)");
    fl->cross_mode = mode;
    fl->mv_dirty = true;
    fl->geom_version++;
    return SKB_OK;
}

int skb_flow_set_overlap(skb_flow *fl, int on) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_overlap: NULL flow");
    fl->bg.enabled = on != 0;
    return SKB_OK;
}

int skb_flow_set_self_exclusion(skb_flow *fl, int fused) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_self_exclusion: NULL flow");
    fl->self_excl = fused != 0;
    fl->mv_dirty = true;
    fl->geom_version++;
    return SKB_OK;
}

int skb_flow_set_target_window(skb_flow *fl, int64_t begin, int64_t end) {
    if (!fl || begin < 0 || (end >= 0 && end < begin))
        return set_error(SKB_ERR_INVALID, "skb_flow_set_target_window: bad window [%lld, %lld)", (long long)begin,
                         (long long)end);
    fl->win_begin = begin;
    fl->win_end = end;
    fl->use_ranges = false;
    fl->mv_dirty = true;
    fl->ops_ready = false; // resident fiber operators belong to one set of fiber rows
    fl->geom_version++;
    return SKB_OK;
}

int skb_flow_set_target_ranges(skb_flow *fl, int fiber_begin, int fiber_end, int64_t shell_begin, int64_t shell_end,
                               int64_t body_begin, int64_t body_end) {
    if (!fl || fiber_begin < 0 || fiber_end < fiber_begin || shell_begin < 0 || shell_end < shell_begin ||
        body_begin < 0 || body_end < body_begin)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_target_ranges: bad ranges");
    fl->rq_f0 = fiber_begin;
    fl->rq_f1 = fiber_end;
    fl->rq_s0 = shell_begin;
    fl->rq_s1 = shell_end;
    fl->rq_b0 = body_begin;
    fl->rq_b1 = body_end;
    fl->use_ranges = true;
    fl->mv_dirty = true;
    fl->ops_ready = false;
    fl->geom_version++;
    return SKB_OK;
}

int skb_flow_matvec(skb_flow *fl, const double *fib_forces, const double *shell_density, const double *body_densities,
                    const double *body_forces_torques, double eta, double *v_all) {
    if (!fl || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_matvec: bad arguments");
    const long long nf = fl->n_fib, ns = fl->n_shell, nb = fl->n_body, n_all = nf + ns + nb;
    if ((nf > 0 && !fib_forces) || (ns > 0 && !shell_density) || (nb > 0 && !body_densities) ||
        (fl->n_bodies > 0 && !body_forces_torques) || (n_all > 0 && !v_all))
        return set_error(SKB_ERR_INVALID, "skb_flow_matvec: NULL input for a non-empty class");
    SKB_TRY(begin_call(fl));
    if (n_all == 0)
        return SKB_OK;
    SKB_TRY(prepare_matvec_targets(fl));
    const long long n_win = fl->n_win;
    if (n_win == 0)
        return SKB_OK;
    std::vector<double> f, t;
    if (fl->n_bodies > 0)
        split_forces_torques(body_forces_torques, fl->n_bodies, f, t);
    const HostStrengths in{fib_forces, shell_density, body_densities, f.data(), t.data()};
    const size_t n_out = (size_t)n_win * 3;
    if (fl->graphs_enabled && (n_strengths(fl) + n_out) * 8 <= kGraphMaxBytes) {
        // launch-bound size: stage through pinned memory and replay the whole sequence as one CUDA graph
        HostStrengths staged;
        double *h_v = nullptr;
        SKB_TRY(fill_stage(fl, in, n_out, &staged, &h_v));
        SKB_TRY(fl->vel.ensure((size_t)n_win * 24));
        unsigned long long key = mix_key(fl->geom_version, (unsigned long long)fl->fa);
        key = mix_key(key, (unsigned long long)fl->n_win);
        key = mix_key(key, dbl_bits(eta));
        key = mix_key(key, buffer_key(fl, 1));
        auto body = [&]() -> int {
            SKB_TRY(upload_strengths(fl, staged));
            SKB_TRY(matvec_core(fl, (const double *)fl->in_fib.ptr, (const double *)fl->in_shell.ptr,
                                (const double *)fl->in_body.ptr, (const double *)fl->in_force.ptr,
                                (const double *)fl->in_torque.ptr, eta, (double *)fl->vel.ptr));
            CUDA_TRY(cudaMemcpyAsync(h_v, fl->vel.ptr, (size_t)n_win * 24, cudaMemcpyDeviceToHost, fl->stream));
            return SKB_OK;
        };
        SKB_TRY(host_call_start(fl));
        CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
        SKB_TRY(run_graphed(fl, fl->g_matvec, key, body));
        CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
        SKB_TRY(host_call_finish(fl));
        std::memcpy(v_all, h_v, (size_t)n_win * 24);
        return SKB_OK;
    }
    SKB_TRY(host_call_start(fl));
    SKB_TRY(upload_strengths(fl, in));
    SKB_TRY(fl->vel.ensure((size_t)n_win * 24));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(matvec_core(fl, (const double *)fl->in_fib.ptr, (const double *)fl->in_shell.ptr,
                        (const double *)fl->in_body.ptr, (const double *)fl->in_force.ptr,
                        (const double *)fl->in_torque.ptr, eta, (double *)fl->vel.ptr));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(v_all, fl->vel.ptr, (size_t)n_win * 24, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl);
}

int skb_flow_matvec_device(skb_flow *fl, const double *d_fib_forces, const double *d_shell_density,
                           const double *d_body_densities, const double *d_body_forces, const double *d_body_torques,
                           double eta, double *d_v_window, void *stream) {
    if (!fl || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_matvec_device: bad arguments");
    const long long nf = fl->n_fib, ns = fl->n_shell, nb = fl->n_body, n_all = nf + ns + nb;
    if ((nf > 0 && !d_fib_forces) || (ns > 0 && !d_shell_density) || (nb > 0 && !d_body_densities) ||
        (fl->n_bodies > 0 && (!d_body_forces || !d_body_torques)))
        return set_error(SKB_ERR_INVALID, "skb_flow_matvec_device: NULL input for a non-empty class");
    SKB_TRY(begin_call(fl));
    if (n_all == 0)
        return SKB_OK;
    SKB_TRY(prepare_matvec_targets(fl));
    if (fl->n_win > 0 && !d_v_window)
        return set_error(SKB_ERR_INVALID, "skb_flow_matvec_device: NULL output");
    fl->cur = (cudaStream_t)stream;
    SKB_TRY(matvec_core(fl, d_fib_forces, d_shell_density, d_body_densities, d_body_forces, d_body_torques, eta,
                        d_v_window));
    return device_call_finish(fl);
}

// ---- per-fiber dense operators (SURVEY.md §8f N2) ---------------------------------------------------------------

int skb_flow_set_fiber_class(skb_flow *fl, int n_nodes, const double *D_1_0, const double *P_downsample_bc) {
    if (!fl || !D_1_0 || !P_downsample_bc)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_class: NULL argument");
    if (n_nodes < 4) // bc_start_i = 4n - 14 must leave room for the 14 boundary rows (ffd.cpp:279)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_class: n_nodes = %d (need >= 4)", n_nodes);
    const size_t n = (size_t)n_nodes;
    skb_flow::FiberClass &c = fl->fiber_classes[n_nodes];
    c.D.assign(D_1_0, D_1_0 + n * n);
    c.P.assign(P_downsample_bc, P_downsample_bc + (4 * n - 14) * 4 * n);
    fl->ops_ready = false;
    return SKB_OK;
}

int skb_flow_set_fiber_operators(skb_flow *fl, const double *A, const double *force_operator, const double *xs,
                                 const double *length_prev, const int *plus_bc_velocity) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_operators: NULL flow");
    fl->ops_ready = false;
    CUDA_TRY(cudaSetDevice(fl->dev));
    // the resident operators are those of the fibers whose rows are in this flow's target list: all of them, or the
    // rank's own fibers under skb_flow_set_target_ranges / an aligned skb_flow_set_target_window
    SKB_TRY(prepare_matvec_targets(fl));
    int f0 = 0, f1 = 0;
    if (fl->n_fibers > 0) {
        const auto &off = fl->h_fiber_off;
        f0 = (int)(std::lower_bound(off.begin(), off.end(), fl->fa) - off.begin());
        f1 = (int)(std::lower_bound(off.begin(), off.end(), fl->fb) - off.begin());
        if (off[(size_t)f0] != fl->fa || off[(size_t)f1] != fl->fb)
            return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_operators: the target window [%lld, %lld) cuts a "
                                              "fiber; use skb_flow_set_target_ranges (whole fibers)", fl->fa, fl->fb);
    }
    fl->op_f0 = f0;
    fl->op_f1 = f1;
    const int nfib = f1 - f0;
    if (nfib == 0) {
        fl->n_items_A = fl->n_items_F = 0;
        fl->ops_ready = true;
        return SKB_OK;
    }
    if (!A || !force_operator || !xs || !length_prev || !plus_bc_velocity)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_operators: NULL argument");
    // class matrices -> one device buffer, per-fiber offsets into it; per class also the non-zero column range of every
    // row of P_downsample_bc (block diagonal in the reference, ffd.cpp:551-555: the kernel walks the range only)
    std::vector<double> h_class;
    std::vector<int2> h_ranges;
    std::map<int, std::pair<long long, long long>> class_off;
    std::map<int, long long> range_off;
    for (const auto &kv : fl->fiber_classes) {
        class_off[kv.first] = {(long long)h_class.size(), (long long)(h_class.size() + kv.second.D.size())};
        h_class.insert(h_class.end(), kv.second.D.begin(), kv.second.D.end());
        h_class.insert(h_class.end(), kv.second.P.begin(), kv.second.P.end());
        const int nn = kv.first, bc = 4 * nn - 14;
        range_off[nn] = (long long)h_ranges.size();
        for (int r = 0; r < bc; ++r) {
            int c0 = 4 * nn, c1 = 0;
            for (int c = 0; c < 4 * nn; ++c)
                if (kv.second.P[(size_t)c * bc + r] != 0.0) {
                    c0 = std::min(c0, c);
                    c1 = c + 1;
                }
            h_ranges.push_back(c1 > c0 ? make_int2(c0, c1) : make_int2(0, 0));
        }
        for (int j = 0; j < nn; ++j) { // D_1_0 (n x n, column-major): non-zero row range of every column (banded)
            int i0 = nn, i1 = 0;
            for (int i = 0; i < nn; ++i)
                if (kv.second.D[(size_t)j * nn + i] != 0.0) {
                    i0 = std::min(i0, i);
                    i1 = i + 1;
                }
            h_ranges.push_back(i1 > i0 ? make_int2(i0, i1) : make_int2(0, 0));
        }
    }
    std::vector<long long> cD((size_t)nfib), cP((size_t)nfib), cR((size_t)nfib);
    std::vector<FiberGemvItem> itA, itF;
    long long offA = 0, offF = 0;
    int max_n = 0;
    const long long node0 = fl->h_fiber_off[(size_t)f0]; // x / fw / v / res of the own fibers are indexed from here
    for (int f = 0; f < nfib; ++f) {
        const int n = fl->h_fiber_n[(size_t)(f0 + f)];
        auto it = class_off.find(n);
        if (it == class_off.end())
            return set_error(SKB_ERR_INVALID, "fiber %d has %d nodes but skb_flow_set_fiber_class(%d, ...) was never "
                                              "called", f0 + f, n, n);
        if (!(length_prev[f] > 0))
            return set_error(SKB_ERR_INVALID, "fiber %d: length_prev = %g", f0 + f, length_prev[f]);
        cD[f] = it->second.first;
        cP[f] = it->second.second;
        cR[f] = range_off[n];
        max_n = std::max(max_n, n);
        const long long node_off = fl->h_fiber_off[(size_t)(f0 + f)] - node0;
        for (int r0 = 0; r0 < 4 * n; r0 += kFiberGemvRows)
            itA.push_back(FiberGemvItem{offA, 4 * node_off, 4 * node_off, 4 * n, 4 * n, r0, n, f, 0});
        for (int r0 = 0; r0 < 3 * n; r0 += kFiberGemvRows)
            itF.push_back(FiberGemvItem{offF, 4 * node_off, node_off, 3 * n, 4 * n, r0, n, f, 0});
        offA += 16LL * n * n;
        offF += 12LL * n * n;
    }
    // x (4n) + slice partials + vT (4n) + s (n)
    fl->gemv_smem = ((size_t)2 * ((4 * max_n + 1) & ~1) + kFiberGemvThreads + (size_t)max_n) * sizeof(double);
    if (fl->gemv_smem > 200 * 1024)
        return set_error(SKB_ERR_INVALID, "fiber with %d nodes exceeds the shared-memory fiber operator kernels", max_n);
    if (fl->gemv_smem > 48 * 1024) {
        CUDA_TRY(cudaFuncSetAttribute(fiber_gemv_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)fl->gemv_smem));
        CUDA_TRY(cudaFuncSetAttribute(fiber_gemv_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)fl->gemv_smem));
        CUDA_TRY(cudaFuncSetAttribute(fiber_gemv_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)fl->gemv_smem));
    }
    const long long nf = fl->fb - fl->fa; // nodes of the own fibers
    auto put = [&](DevBuf &b, const void *h, size_t bytes) -> int {
        SKB_TRY(b.ensure(bytes));
        CUDA_TRY(cudaMemcpyAsync(b.ptr, h, bytes, cudaMemcpyHostToDevice, fl->stream));
        return SKB_OK;
    };
    SKB_TRY(fl->op_A.ensure((size_t)offA * 8));
    SKB_TRY(fl->op_F.ensure((size_t)offF * 8));
    SKB_TRY(upload_pageable(fl->op_A.ptr, A, (size_t)offA * 8, fl->stream));
    SKB_TRY(upload_pageable(fl->op_F.ptr, force_operator, (size_t)offF * 8, fl->stream));
    SKB_TRY(put(fl->op_xs, xs, (size_t)nf * 24));
    SKB_TRY(put(fl->op_len, length_prev, (size_t)nfib * 8));
    SKB_TRY(put(fl->op_plus, plus_bc_velocity, (size_t)nfib * sizeof(int)));
    SKB_TRY(put(fl->op_class, h_class.data(), h_class.size() * 8));
    SKB_TRY(put(fl->op_classD, cD.data(), cD.size() * 8));
    SKB_TRY(put(fl->op_classP, cP.data(), cP.size() * 8));
    SKB_TRY(put(fl->op_classR, cR.data(), cR.size() * 8));
    SKB_TRY(put(fl->op_ranges, h_ranges.data(), h_ranges.size() * sizeof(int2)));
    SKB_TRY(put(fl->items_A, itA.data(), itA.size() * sizeof(FiberGemvItem)));
    SKB_TRY(put(fl->items_F, itF.data(), itF.size() * sizeof(FiberGemvItem)));
    SKB_TRY(fl->x_fib.ensure((size_t)nf * 32));
    SKB_TRY(fl->res_fib.ensure((size_t)nf * 32));
    SKB_TRY(fl->vb.ensure((size_t)nfib * 56));
    CUDA_TRY(cudaStreamSynchronize(fl->stream)); // the host vectors above go out of scope
    fl->n_items_A = (int)itA.size();
    fl->n_items_F = (int)itF.size();
    fl->op_A_elems = offA;
    fl->ops_gen++;
    fl->ops_ready = true;
    return SKB_OK;
}

int skb_flow_set_fiber_preconditioner(skb_flow *fl, const double *A_inv) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_preconditioner: NULL flow");
    if (!fl->ops_ready)
        return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_preconditioner: call skb_flow_set_fiber_operators "
                                          "first (it defines the fibers and their order)");
    if (fl->op_A_elems > 0) {
        if (!A_inv)
            return set_error(SKB_ERR_INVALID, "skb_flow_set_fiber_preconditioner: NULL argument");
        CUDA_TRY(cudaSetDevice(fl->dev));
        SKB_TRY(fl->op_Ainv.ensure((size_t)fl->op_A_elems * 8));
        SKB_TRY(upload_pageable(fl->op_Ainv.ptr, A_inv, (size_t)fl->op_A_elems * 8, fl->stream));
    }
    fl->precond_gen = fl->ops_gen;
    return SKB_OK;
}

int skb_flow_apply_fiber_preconditioner(skb_flow *fl, const double *x_fibers, double *y) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_preconditioner: NULL flow");
    SKB_TRY(need_precond(fl, "skb_flow_apply_fiber_preconditioner"));
    const long long nf = fl->fb - fl->fa;
    SKB_TRY(begin_call(fl));
    if (nf == 0)
        return SKB_OK;
    if (!x_fibers || !y)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_preconditioner: NULL argument");
    SKB_TRY(host_call_start(fl));
    CUDA_TRY(cudaMemcpyAsync(fl->x_fib.ptr, x_fibers, (size_t)nf * 32, cudaMemcpyHostToDevice, fl->stream));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(fiber_precond_dev(fl, (const double *)fl->x_fib.ptr, (double *)fl->res_fib.ptr));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(y, fl->res_fib.ptr, (size_t)nf * 32, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl);
}

int skb_flow_apply_fiber_preconditioner_device(skb_flow *fl, const double *d_x_fibers, double *d_y, void *stream) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_preconditioner_device: NULL flow");
    SKB_TRY(need_precond(fl, "skb_flow_apply_fiber_preconditioner_device"));
    SKB_TRY(begin_call(fl));
    if (fl->n_items_A == 0)
        return SKB_OK;
    if (!d_x_fibers || !d_y)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_preconditioner_device: NULL argument");
    fl->cur = (cudaStream_t)stream;
    SKB_TRY(fiber_precond_dev(fl, d_x_fibers, d_y));
    return device_call_finish(fl);
}

int skb_flow_apply_fiber_force(skb_flow *fl, const double *x_fibers, double *fw) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_force: NULL flow");
    SKB_TRY(need_ops(fl, "skb_flow_apply_fiber_force"));
    const long long nf = fl->fb - fl->fa; // nodes of the own fibers (all of them without a window)
    SKB_TRY(begin_call(fl));
    if (nf == 0)
        return SKB_OK;
    if (!x_fibers || !fw)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_force: NULL argument");
    SKB_TRY(host_call_start(fl));
    CUDA_TRY(cudaMemcpyAsync(fl->x_fib.ptr, x_fibers, (size_t)nf * 32, cudaMemcpyHostToDevice, fl->stream));
    SKB_TRY(fl->in_fib.ensure((size_t)nf * 24));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(fiber_force_dev(fl, (const double *)fl->x_fib.ptr, (double *)fl->in_fib.ptr));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(fw, fl->in_fib.ptr, (size_t)nf * 24, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl);
}

int skb_flow_fiber_matvec(skb_flow *fl, const double *x_fibers, const double *v_fibers, const double *v_fib_boundary,
                          double *res) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_fiber_matvec: NULL flow");
    SKB_TRY(need_ops(fl, "skb_flow_fiber_matvec"));
    const long long nf = fl->fb - fl->fa;
    SKB_TRY(begin_call(fl));
    if (nf == 0)
        return SKB_OK;
    if (!x_fibers || !v_fibers || !res)
        return set_error(SKB_ERR_INVALID, "skb_flow_fiber_matvec: NULL argument");
    SKB_TRY(host_call_start(fl));
    CUDA_TRY(cudaMemcpyAsync(fl->x_fib.ptr, x_fibers, (size_t)nf * 32, cudaMemcpyHostToDevice, fl->stream));
    SKB_TRY(fl->vel.ensure((size_t)nf * 24));
    CUDA_TRY(cudaMemcpyAsync(fl->vel.ptr, v_fibers, (size_t)nf * 24, cudaMemcpyHostToDevice, fl->stream));
    if (v_fib_boundary)
        CUDA_TRY(cudaMemcpyAsync(fl->vb.ptr, v_fib_boundary, (size_t)(fl->op_f1 - fl->op_f0) * 56, cudaMemcpyHostToDevice,
                                 fl->stream));
    CUDA_TRY(cudaEventRecord(fl->ev0, fl->stream));
    SKB_TRY(fiber_matvec_dev(fl, (const double *)fl->x_fib.ptr, (const double *)fl->vel.ptr,
                             v_fib_boundary ? (const double *)fl->vb.ptr : nullptr, (double *)fl->res_fib.ptr));
    CUDA_TRY(cudaEventRecord(fl->ev1, fl->stream));
    CUDA_TRY(cudaMemcpyAsync(res, fl->res_fib.ptr, (size_t)nf * 32, cudaMemcpyDeviceToHost, fl->stream));
    return host_call_finish(fl);
}

int skb_flow_apply_fiber_force_device(skb_flow *fl, const double *d_x_fibers, double *d_fw, void *stream) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_force_device: NULL flow");
    SKB_TRY(need_ops(fl, "skb_flow_apply_fiber_force_device"));
    SKB_TRY(begin_call(fl));
    if (fl->n_items_F == 0)
        return SKB_OK;
    if (!d_x_fibers || !d_fw)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_fiber_force_device: NULL argument");
    fl->cur = (cudaStream_t)stream;
    SKB_TRY(fiber_force_dev(fl, d_x_fibers, d_fw));
    return device_call_finish(fl);
}

int skb_flow_fiber_matvec_device(skb_flow *fl, const double *d_x_fibers, const double *d_v_fibers,
                                 const double *d_v_fib_boundary, double *d_res, void *stream) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_fiber_matvec_device: NULL flow");
    SKB_TRY(need_ops(fl, "skb_flow_fiber_matvec_device"));
    SKB_TRY(begin_call(fl));
    if (fl->n_items_A == 0)
        return SKB_OK;
    if (!d_x_fibers || !d_v_fibers || !d_res)
        return set_error(SKB_ERR_INVALID, "skb_flow_fiber_matvec_device: NULL argument");
    fl->cur = (cudaStream_t)stream;
    SKB_TRY(fiber_matvec_dev(fl, d_x_fibers, d_v_fibers, d_v_fib_boundary, d_res));
    return device_call_finish(fl);
}

int skb_flow_apply_matvec(skb_flow *fl, const double *x_fibers, const double *shell_density,
                          const double *body_densities, const double *body_forces_torques,
                          const double *fiber_link_conditions, double eta, double *res_fibers, double *v_shell,
                          double *v_bodies) {
    return apply_matvec_impl(fl, nullptr, x_fibers, shell_density, body_densities, body_forces_torques,
                             fiber_link_conditions, eta, res_fibers, v_shell, v_bodies);
}

int skb_flow_apply_matvec_dense(skb_flow *fl, skb_dense *dn, const double *x_fibers, const double *x_shell,
                                const double *body_densities, const double *body_forces_torques,
                                const double *fiber_link_conditions, double eta, double *res_fibers,
                                double *res_shell, double *v_bodies) {
    if (!fl || !dn)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_matvec_dense: NULL handle");
    SKB_TRY(check_dense_handle(fl, dn, "skb_flow_apply_matvec_dense"));
    return apply_matvec_impl(fl, dn, x_fibers, x_shell, body_densities, body_forces_torques, fiber_link_conditions,
                             eta, res_fibers, res_shell, v_bodies);
}

int skb_flow_apply_matvec_device(skb_flow *fl, skb_dense *dn, const double *d_x_fibers, const double *d_x_shell,
                                 const double *d_body_densities, const double *d_body_forces,
                                 const double *d_body_torques, const double *d_fiber_link_conditions, double eta,
                                 double *d_res_fibers, double *d_out_shell, double *d_v_bodies, void *stream) {
    if (!fl || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_matvec_device: bad arguments");
    SKB_TRY(need_ops(fl, "skb_flow_apply_matvec_device"));
    SKB_TRY(begin_call(fl));
    SKB_TRY(prepare_matvec_targets(fl));
    if (dn)
        SKB_TRY(check_dense_handle(fl, dn, "skb_flow_apply_matvec_device"));
    const long long n_fw = fl->fb - fl->fa, n_sw = fl->sb - fl->sa, n_bw = fl->bb - fl->ba;
    if ((n_fw > 0 && (!d_x_fibers || !d_res_fibers)) || (n_sw > 0 && (!d_x_shell || !d_out_shell)) ||
        (fl->n_body > 0 && !d_body_densities) || (n_bw > 0 && !d_v_bodies) ||
        (fl->n_bodies > 0 && (!d_body_forces || !d_body_torques)))
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_matvec_device: NULL argument for a non-empty class");
    if (fl->grp.size == 1 && fl->n_win == 0)
        return SKB_OK;
    if (fl->grp.size == 1 && fl->n_win != fl->n_fib + fl->n_shell + fl->n_body)
        return set_error(SKB_ERR_INVALID, "skb_flow_apply_matvec_device: a flow that owns only part of the rows must be a "
                                          "group member (skb_flow_group_init): the fiber forces of the other rows' "
                                          "fibers have to come from somewhere");
    fl->cur = (cudaStream_t)stream;
    SKB_TRY(apply_matvec_core(fl, dn, d_x_fibers, d_x_shell, d_body_densities, d_body_forces, d_body_torques,
                              d_fiber_link_conditions, eta, d_res_fibers, d_out_shell, d_v_bodies));
    return device_call_finish(fl);
}

int skb_flow_last_sym_kernel(const skb_flow *fl, double *ms, int64_t *pairs) {
    if (!fl)
        return set_error(SKB_ERR_INVALID, "skb_flow_last_sym_kernel: NULL");
    return skb_ctx_last_sym_kernel(fl->fib[1], ms, pairs);
}

int skb_flow_last_stats(const skb_flow *fl, skb_flow_stats *out) {
    if (!fl || !out)
        return set_error(SKB_ERR_INVALID, "skb_flow_last_stats: NULL");
    *out = fl->stats;
    return SKB_OK;
}

// ---- skb_mflow ---------------------------------------------------------------------------------------------------

int skb_mflow_create(const int *devices, int n, skb_mflow **out) {
    if (!out || n < 1 || n > kMaxGroup)
        return set_error(SKB_ERR_INVALID, "skb_mflow_create: need 1 <= n <= %d devices", kMaxGroup);
    *out = nullptr;
    std::unique_ptr<skb_mflow> mf(new skb_mflow);
    mf->n = n;
    mf->m.assign(n, nullptr);
    mf->dn.assign(n, nullptr);
    mf->io.resize(n);
    for (int g = 0; g < n; ++g) {
        mf->devs.push_back(devices ? devices[g] : g);
        int rc = skb_flow_create(mf->devs[g], &mf->m[g]);
        if (rc == SKB_OK) {
            cudaSetDevice(mf->devs[g]);
            if (cudaEventCreate(&mf->io[g].e0) != cudaSuccess || cudaEventCreate(&mf->io[g].e1) != cudaSuccess)
                rc = set_error(SKB_ERR_CUDA, "cudaEventCreate failed");
        }
        if (rc != SKB_OK) {
            for (int h = 0; h <= g; ++h)
                skb_flow_destroy(mf->m[h]);
            return rc;
        }
    }
    mf->workers.reset(new Workers(n));
    *out = mf.release();
    return SKB_OK;
}

int skb_mflow_destroy(skb_mflow *mf) {
    if (!mf)
        return SKB_OK;
    mf->workers.reset();
    for (int g = 0; g < mf->n; ++g) {
        cudaSetDevice(mf->devs[g]);
        cudaDeviceSynchronize();
    }
    for (int g = 0; g < mf->n; ++g) {
        cudaSetDevice(mf->devs[g]);
        skb_mflow::IO &io = mf->io[g];
        DevBuf *bufs[] = {&io.x, &io.xs, &io.bd, &io.f, &io.t, &io.link, &io.res, &io.outs, &io.vb, &io.ff, &io.v};
        for (DevBuf *b : bufs)
            b->release();
        if (io.e0) cudaEventDestroy(io.e0);
        if (io.e1) cudaEventDestroy(io.e1);
        skb_dense_destroy(mf->dn[g]);
        skb_flow_destroy(mf->m[g]);
    }
    delete mf;
    return SKB_OK;
}

int skb_mflow_n_devices(const skb_mflow *mf, int *n) {
    if (!mf || !n)
        return set_error(SKB_ERR_INVALID, "skb_mflow_n_devices: NULL");
    *n = mf->n;
    return SKB_OK;
}

int skb_mflow_set_fibers(skb_mflow *mf, const double *r_fib, const int *n_nodes, const double *length, int n_fibers) {
    if (!mf || n_fibers < 0)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_fibers: bad arguments");
    std::vector<long long> off((size_t)n_fibers + 1, 0);
    for (int f = 0; f < n_fibers; ++f)
        off[(size_t)f + 1] = off[(size_t)f] + (n_nodes ? n_nodes[f] : 0);
    const bool resized = off != mf->fiber_off;
    SKB_TRY(mf->workers->run([&](int g) -> int { return skb_flow_set_fibers(mf->m[g], r_fib, n_nodes, length, n_fibers); }));
    mf->n_fibers = n_fibers;
    mf->n_fib = off[(size_t)n_fibers];
    mf->fiber_off = off;
    mf->fiber_n.assign(n_nodes, n_nodes + n_fibers);
    mf->ops_ready = false;
    if (resized)
        mf->part_dirty = true;
    return SKB_OK;
}

int skb_mflow_set_periphery(skb_mflow *mf, const double *node_pos, const double *node_normal, int64_t n_nodes) {
    if (!mf || n_nodes < 0)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_periphery: bad arguments");
    SKB_TRY(mf->workers->run([&](int g) -> int { return skb_flow_set_periphery(mf->m[g], node_pos, node_normal, n_nodes); }));
    if (mf->n_shell != n_nodes)
        mf->part_dirty = true;
    mf->n_shell = n_nodes;
    return SKB_OK;
}

int skb_mflow_set_bodies(skb_mflow *mf, const double *node_pos, const double *node_normal, int64_t n_nodes,
                         const double *centers, int n_bodies) {
    if (!mf || n_nodes < 0 || n_bodies < 0)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_bodies: bad arguments");
    SKB_TRY(mf->workers->run(
        [&](int g) { return skb_flow_set_bodies(mf->m[g], node_pos, node_normal, n_nodes, centers, n_bodies); }));
    if (mf->n_body != n_nodes)
        mf->part_dirty = true;
    mf->n_body = n_nodes;
    mf->n_bodies = n_bodies;
    return SKB_OK;
}

int skb_mflow_set_cross(skb_mflow *mf, int mode) {
    if (!mf)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_cross: NULL");
    for (int g = 0; g < mf->n; ++g)
        SKB_TRY(skb_flow_set_cross(mf->m[g], mode));
    mf->part_dirty = true; // the members' target lists change: re-run the warm-up
    return SKB_OK;
}

int skb_mflow_set_overlap(skb_mflow *mf, int on) {
    if (!mf)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_overlap: NULL");
    for (int g = 0; g < mf->n; ++g)
        SKB_TRY(skb_flow_set_overlap(mf->m[g], on));
    return SKB_OK;
}

int skb_mflow_set_self_exclusion(skb_mflow *mf, int fused) {
    if (!mf)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_self_exclusion: NULL");
    for (int g = 0; g < mf->n; ++g)
        SKB_TRY(skb_flow_set_self_exclusion(mf->m[g], fused));
    return SKB_OK;
}

int skb_mflow_partition(skb_mflow *mf, int member, int *fiber_begin, int *fiber_end, int64_t *shell_begin,
                        int64_t *shell_end, int64_t *body_begin, int64_t *body_end) {
    if (!mf || member < 0 || member >= mf->n)
        return set_error(SKB_ERR_INVALID, "skb_mflow_partition: bad member");
    SKB_TRY(mflow_prepare(mf));
    if (fiber_begin) *fiber_begin = mf->f0[member];
    if (fiber_end) *fiber_end = mf->f1[member];
    if (shell_begin) *shell_begin = mf->s0[member];
    if (shell_end) *shell_end = mf->s1[member];
    if (body_begin) *body_begin = mf->b0[member];
    if (body_end) *body_end = mf->b1[member];
    return SKB_OK;
}

// host-only (no GPU needed): the partition skb_mflow uses, for rank-per-GPU hosts that want the same one
int skb_partition_query(const int *n_nodes, int n_fibers, int64_t n_shell, int64_t n_body, int n_members, int member,
                        int64_t *out6) {
    if (n_fibers < 0 || (n_fibers > 0 && !n_nodes) || n_shell < 0 || n_body < 0 || n_members < 1 || member < 0 ||
        member >= n_members || !out6)
        return set_error(SKB_ERR_INVALID, "skb_partition_query: bad arguments");
    std::vector<long long> off((size_t)n_fibers + 1, 0);
    for (int f = 0; f < n_fibers; ++f)
        off[(size_t)f + 1] = off[(size_t)f] + n_nodes[f];
    std::vector<int> f0, f1;
    std::vector<long long> s0, s1, b0, b1;
    partition_rows(off, n_shell, n_body, n_members, f0, f1, s0, s1, b0, b1);
    out6[0] = f0[member], out6[1] = f1[member], out6[2] = s0[member], out6[3] = s1[member], out6[4] = b0[member],
    out6[5] = b1[member];
    return SKB_OK;
}

int skb_mflow_set_fiber_class(skb_mflow *mf, int n_nodes, const double *D_1_0, const double *P_downsample_bc) {
    if (!mf)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_fiber_class: NULL");
    for (int g = 0; g < mf->n; ++g)
        SKB_TRY(skb_flow_set_fiber_class(mf->m[g], n_nodes, D_1_0, P_downsample_bc));
    mf->ops_ready = false;
    return SKB_OK;
}

int skb_mflow_set_fiber_operators(skb_mflow *mf, const double *A, const double *force_operator, const double *xs,
                                  const double *length_prev, const int *plus_bc_velocity) {
    if (!mf)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_fiber_operators: NULL");
    SKB_TRY(mflow_prepare(mf));
    if (mf->n_fibers > 0 && (!A || !force_operator || !xs || !length_prev || !plus_bc_velocity))
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_fiber_operators: NULL argument");
    SKB_TRY(mf->workers->run([&](int g) -> int {
        const int f0 = mf->f0[g];
        if (mf->f1[g] == f0)
            return skb_flow_set_fiber_operators(mf->m[g], nullptr, nullptr, nullptr, nullptr, nullptr);
        return skb_flow_set_fiber_operators(mf->m[g], A + op_offset(mf, f0, 4), force_operator + op_offset(mf, f0, 3),
                                            xs + 3 * mf->fiber_off[(size_t)f0], length_prev + f0, plus_bc_velocity + f0);
    }));
    mf->ops_ready = true;
    return SKB_OK;
}

int skb_mflow_set_fiber_preconditioner(skb_mflow *mf, const double *A_inv) {
    if (!mf || !mf->ops_ready)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_fiber_preconditioner: call skb_mflow_set_fiber_operators first");
    return mf->workers->run([&](int g) -> int {
        const int f0 = mf->f0[g];
        return skb_flow_set_fiber_preconditioner(mf->m[g], mf->f1[g] == f0 ? nullptr : A_inv + op_offset(mf, f0, 4));
    });
}

// the periphery's dense operator, rows block-partitioned like the periphery rows (periphery.cpp:387-417)
int skb_mflow_set_dense(skb_mflow *mf, int op, const double *A_rowmajor, int64_t n_rows, int64_t n_cols) {
    if (!mf || !A_rowmajor || n_rows != 3 * mf->n_shell || n_cols != 3 * mf->n_shell)
        return set_error(SKB_ERR_INVALID, "skb_mflow_set_dense: need the (3 N_s) x (3 N_s) operator of the %lld periphery "
                                          "nodes set before", mf ? mf->n_shell : 0LL);
    SKB_TRY(mflow_prepare(mf));
    SKB_TRY(mf->workers->run([&](int g) -> int {
        if (!mf->dn[g])
            SKB_TRY(skb_dense_create_on(&mf->devs[g], 1, &mf->dn[g]));
        return skb_dense_set_matrix(mf->dn[g], op, A_rowmajor + (size_t)(3 * mf->s0[g]) * (size_t)n_cols,
                                    3 * (mf->s1[g] - mf->s0[g]), n_cols);
    }));
    if (op == SKB_DENSE_STRESSLET_PLUS_COMPLEMENTARY)
        mf->has_dense = true;
    return SKB_OK;
}

// v_all over [fibers | periphery | bodies] like skb_flow_matvec; complete host arrays in and out
int skb_mflow_matvec(skb_mflow *mf, const double *fib_forces, const double *shell_density, const double *body_densities,
                     const double *body_forces_torques, double eta, double *v_all) {
    if (!mf || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_mflow_matvec: bad arguments");
    const long long nf = mf->n_fib, ns = mf->n_shell, nb = mf->n_body;
    if ((nf > 0 && !fib_forces) || (ns > 0 && !shell_density) || (nb > 0 && !body_densities) ||
        (mf->n_bodies > 0 && !body_forces_torques) || (nf + ns + nb > 0 && !v_all))
        return set_error(SKB_ERR_INVALID, "skb_mflow_matvec: NULL input for a non-empty class");
    SKB_TRY(mflow_prepare(mf));
    std::vector<double> f, t;
    if (mf->n_bodies > 0)
        split_forces_torques(body_forces_torques, mf->n_bodies, f, t);
    SKB_TRY(mflow_size_io(mf, f.size()));
    SKB_TRY(mf->workers->run([&](int g) -> int {
        skb_flow *fl = mf->m[g];
        skb_mflow::IO &io = mf->io[g];
        CUDA_TRY(cudaSetDevice(mf->devs[g]));
        const MemberRows r = member_rows(mf, g);
        const long long a = r.a, n_fw = r.n_fw, n_sw = r.n_sw, n_bw = r.n_bw;
        cudaStream_t st = fl->stream;
        // (mflow_size_io sized every buffer)
        SKB_TRY(upload(fl, io.ff, fib_forces ? fib_forces + 3 * a : nullptr, (size_t)n_fw * 3));
        SKB_TRY(upload(fl, io.xs, shell_density ? shell_density + 3 * mf->s0[g] : nullptr, (size_t)n_sw * 3));
        SKB_TRY(upload(fl, io.bd, body_densities, (size_t)nb * 3));
        SKB_TRY(upload(fl, io.f, f.data(), f.size()));
        SKB_TRY(upload(fl, io.t, t.data(), t.size()));
        SKB_TRY(io.v.ensure((size_t)(n_fw + n_sw + n_bw) * 24 + 8));
        CUDA_TRY(cudaEventRecord(io.e0, st));
        SKB_TRY(skb_flow_matvec_device(fl, (const double *)io.ff.ptr, (const double *)io.xs.ptr,
                                       (const double *)io.bd.ptr, (const double *)io.f.ptr, (const double *)io.t.ptr, eta,
                                       (double *)io.v.ptr, st));
        CUDA_TRY(cudaEventRecord(io.e1, st));
        double *d_v = (double *)io.v.ptr;
        if (n_fw)
            CUDA_TRY(cudaMemcpyAsync(v_all + 3 * a, d_v, (size_t)n_fw * 24, cudaMemcpyDeviceToHost, st));
        if (n_sw)
            CUDA_TRY(cudaMemcpyAsync(v_all + 3 * (nf + mf->s0[g]), d_v + 3 * n_fw, (size_t)n_sw * 24,
                                     cudaMemcpyDeviceToHost, st));
        if (n_bw)
            CUDA_TRY(cudaMemcpyAsync(v_all + 3 * (nf + ns + mf->b0[g]), d_v + 3 * (n_fw + n_sw), (size_t)n_bw * 24,
                                     cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        return SKB_OK;
    }));
    return mflow_collect_stats(mf);
}

// System::apply_matvec (system.cpp:269-324) over n devices: complete host arrays in and out.  out_shell = res_shell
// when skb_mflow_set_dense(SKB_DENSE_STRESSLET_PLUS_COMPLEMENTARY) was called, else v_shell.
int skb_mflow_apply_matvec(skb_mflow *mf, const double *x_fibers, const double *x_shell, const double *body_densities,
                           const double *body_forces_torques, const double *fiber_link_conditions, double eta,
                           double *res_fibers, double *out_shell, double *v_bodies) {
    if (!mf || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_mflow_apply_matvec: bad arguments");
    if (!mf->ops_ready)
        return set_error(SKB_ERR_STATE, "skb_mflow_apply_matvec: call skb_mflow_set_fiber_operators first");
    const long long nf = mf->n_fib, ns = mf->n_shell, nb = mf->n_body;
    if ((nf > 0 && (!x_fibers || !res_fibers)) || (ns > 0 && (!x_shell || !out_shell)) ||
        (nb > 0 && (!body_densities || !v_bodies)) || (mf->n_bodies > 0 && !body_forces_torques))
        return set_error(SKB_ERR_INVALID, "skb_mflow_apply_matvec: NULL argument for a non-empty class");
    SKB_TRY(mflow_prepare(mf));
    std::vector<double> f, t;
    if (mf->n_bodies > 0)
        split_forces_torques(body_forces_torques, mf->n_bodies, f, t);
    SKB_TRY(mflow_size_io(mf, f.size()));
    SKB_TRY(mf->workers->run([&](int g) -> int {
        skb_flow *fl = mf->m[g];
        skb_mflow::IO &io = mf->io[g];
        CUDA_TRY(cudaSetDevice(mf->devs[g]));
        const int f0 = mf->f0[g], f1 = mf->f1[g];
        const MemberRows r = member_rows(mf, g);
        const long long a = r.a, n_fw = r.n_fw, n_sw = r.n_sw, n_bw = r.n_bw;
        cudaStream_t st = fl->stream;
        // (mflow_size_io sized every buffer)
        SKB_TRY(upload(fl, io.x, x_fibers ? x_fibers + 4 * a : nullptr, (size_t)n_fw * 4));
        SKB_TRY(upload(fl, io.xs, x_shell ? x_shell + 3 * mf->s0[g] : nullptr, (size_t)n_sw * 3));
        SKB_TRY(upload(fl, io.bd, body_densities, (size_t)nb * 3));
        SKB_TRY(upload(fl, io.f, f.data(), f.size()));
        SKB_TRY(upload(fl, io.t, t.data(), t.size()));
        SKB_TRY(upload(fl, io.link, fiber_link_conditions ? fiber_link_conditions + 7 * (long long)f0 : nullptr,
                       (size_t)(f1 - f0) * 7));
        SKB_TRY(io.res.ensure((size_t)n_fw * 32 + 8));
        SKB_TRY(io.outs.ensure((size_t)n_sw * 24 + 8));
        SKB_TRY(io.vb.ensure((size_t)n_bw * 24 + 8));
        CUDA_TRY(cudaEventRecord(io.e0, st));
        SKB_TRY(skb_flow_apply_matvec_device(
            fl, mf->has_dense ? mf->dn[g] : nullptr, (const double *)io.x.ptr, (const double *)io.xs.ptr,
            (const double *)io.bd.ptr, (const double *)io.f.ptr, (const double *)io.t.ptr,
            (fiber_link_conditions && f1 > f0) ? (const double *)io.link.ptr : nullptr, eta, (double *)io.res.ptr,
            (double *)io.outs.ptr, (double *)io.vb.ptr, st));
        CUDA_TRY(cudaEventRecord(io.e1, st));
        if (n_fw)
            CUDA_TRY(cudaMemcpyAsync(res_fibers + 4 * a, io.res.ptr, (size_t)n_fw * 32, cudaMemcpyDeviceToHost, st));
        if (n_sw)
            CUDA_TRY(cudaMemcpyAsync(out_shell + 3 * mf->s0[g], io.outs.ptr, (size_t)n_sw * 24, cudaMemcpyDeviceToHost,
                                     st));
        if (n_bw)
            CUDA_TRY(cudaMemcpyAsync(v_bodies + 3 * mf->b0[g], io.vb.ptr, (size_t)n_bw * 24, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        return SKB_OK;
    }));
    return mflow_collect_stats(mf);
}

// System::velocity_at_targets (system.cpp:330-384) over n devices: the targets are block-partitioned, every device
// holds all sources
int skb_mflow_velocity_at_targets(skb_mflow *mf, const double *r_trg, int64_t n_trg, const double *fib_forces,
                                  const double *shell_density, const double *body_densities,
                                  const double *body_forces_torques, double eta, double *vel) {
    if (!mf || n_trg < 0 || (n_trg > 0 && (!r_trg || !vel)) || !(eta > 0))
        return set_error(SKB_ERR_INVALID, "skb_mflow_velocity_at_targets: bad arguments");
    const long long chunk = (n_trg + mf->n - 1) / mf->n;
    SKB_TRY(mf->workers->run([&](int g) -> int {
        const long long b = std::min<long long>(n_trg, g * chunk), e = std::min<long long>(n_trg, (g + 1) * chunk);
        if (e <= b)
            return (int)SKB_OK;
        return skb_flow_velocity_at_targets(mf->m[g], r_trg + 3 * b, e - b, fib_forces, shell_density, body_densities,
                                            body_forces_torques, eta, vel + 3 * b);
    }));
    mflow_sum_stats(mf);
    return SKB_OK;
}

int skb_mflow_last_stats(const skb_mflow *mf, skb_flow_stats *out) {
    if (!mf || !out)
        return set_error(SKB_ERR_INVALID, "skb_mflow_last_stats: NULL");
    *out = mf->stats;
    return SKB_OK;
}

} // extern "C"
