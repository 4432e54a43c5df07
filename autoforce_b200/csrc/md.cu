// Molecular dynamics on the device (include/sgpr_b200.h: sgpr_md_init, sgpr_md_steps): velocity Verlet and BAOAB
// Langevin steps around the prediction step, what ASE's VelocityVerlet / Langevin do around ActiveCalculator in
// prediction mode -- with positions, momenta and forces resident in HBM and no host synchronisation per step.
//
// A step is  drift (B, A[, O, A] into scratch)  ->  prediction of the scratch positions (forces, energy, virial, beta into
// scratch)  ->  kick (B) + commit  ->  finish (thermo row, stop flag, step counter).  Nothing reaches pos/mom/F/beta unless
// the prediction was valid (nl.cu: status[6] = 0), so a step that outgrew the neighbour capacity is never integrated and
// can simply be enqueued again after sizing.  The step counter, the stop step and the invalid flag live on the device:
// the launch arguments are the same every step, and a warm step is captured once into a CUDA graph and replayed.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "sgpr_internal.cuh"

namespace sgpr {
namespace {

constexpr int kMdBlocks = 128;    // fixed grid of the kick kernel: E_kin partials are summed in a fixed order
constexpr int kMdThreads = 256;

struct MdArgs {
    long long N;
    double dt, half_dt, c1, c2, kT, ediff;
    unsigned long long seed;
    int langevin, stop_on_uncertain, init;
    double* pos;
    double* mom;
    const double* mass;
    double* F;
    double* beta;                 // nullptr: no covloss
    double* pos_n;                // scratch of the step in flight
    double* mom_n;
    const double* F_n;
    const double* beta_n;
    const double* ew_n;           // [E, pad, W(9)]
    double* part;                 // [kMdBlocks][2] E_kin and max(beta) partials
    double* thermo;               // [n_steps, 11]
    long long* state;             // {steps done, stop step, invalid, first step of the call}
    const long long* status;      // nl.cu status block: [6] = 1 when the prediction of this step was invalid
};

__device__ __forceinline__ bool md_frozen(const long long* state) { return state[1] >= 0 || state[2] != 0; }

__global__ void md_reset_kernel(long long* state) {
    state[0] = 0;
    state[1] = -1;
    state[2] = 0;
    state[3] = 0;
}

__global__ void md_begin_kernel(long long* state) {
    state[2] = 0;
    state[3] = state[0];
}

// B, A (NVE) or B, A, O, A (Langevin) of ASE's operation order; explicit roundings so that the host loop of numpy
// reproduces it exactly (no contraction into FMA)
__global__ void __launch_bounds__(kMdThreads) md_drift_kernel(MdArgs a) {
    if (md_frozen(a.state)) return;
    const unsigned long long step = (unsigned long long)a.state[0];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.N; i += (long long)gridDim.x * blockDim.x) {
        const double m = a.mass[i];
        double p[3], r[3];
        for (int c = 0; c < 3; ++c) {
            p[c] = __dadd_rn(a.mom[3 * i + c], __dmul_rn(a.half_dt, a.F[3 * i + c]));
            r[c] = a.pos[3 * i + c];
        }
        if (!a.langevin) {
            for (int c = 0; c < 3; ++c) r[c] = __dadd_rn(r[c], __ddiv_rn(__dmul_rn(a.dt, p[c]), m));
        } else {
            double xi[3];
            langevin_normals(a.seed, (uint32_t)i, step, xi);
            const double s = __dmul_rn(a.c2, __dsqrt_rn(__dmul_rn(m, a.kT)));
            for (int c = 0; c < 3; ++c) {
                r[c] = __dadd_rn(r[c], __ddiv_rn(__dmul_rn(a.half_dt, p[c]), m));
                p[c] = __dadd_rn(__dmul_rn(a.c1, p[c]), __dmul_rn(s, xi[c]));
                r[c] = __dadd_rn(r[c], __ddiv_rn(__dmul_rn(a.half_dt, p[c]), m));
            }
        }
        for (int c = 0; c < 3; ++c) {
            a.pos_n[3 * i + c] = r[c];
            a.mom_n[3 * i + c] = p[c];
        }
    }
}

// final B and commit of a valid step (init: commit of the starting forces only); per-block E_kin and max(beta)
__global__ void __launch_bounds__(kMdThreads) md_kick_kernel(MdArgs a) {
    __shared__ double ks[kMdThreads], bs[kMdThreads];
    if (md_frozen(a.state) || a.status[6] != 0) return;
    double ke = 0.0, bmax = -INFINITY;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.N; i += (long long)gridDim.x * blockDim.x) {
        if (!a.init) {
            double p2 = 0.0;
            for (int c = 0; c < 3; ++c) {
                const double p = __dadd_rn(a.mom_n[3 * i + c], __dmul_rn(a.half_dt, a.F_n[3 * i + c]));
                a.mom[3 * i + c] = p;
                a.pos[3 * i + c] = a.pos_n[3 * i + c];
                p2 += p * p;
            }
            ke += 0.5 * p2 / a.mass[i];
        }
        for (int c = 0; c < 3; ++c) a.F[3 * i + c] = a.F_n[3 * i + c];
        if (a.beta) {
            const double b = a.beta_n[i];
            a.beta[i] = b;
            bmax = nan_max(bmax, b);
        }
    }
    ks[threadIdx.x] = ke;
    bs[threadIdx.x] = bmax;
    __syncthreads();
    for (int w = kMdThreads / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            ks[threadIdx.x] += ks[threadIdx.x + w];
            bs[threadIdx.x] = nan_max(bs[threadIdx.x], bs[threadIdx.x + w]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        a.part[2 * blockIdx.x] = ks[0];
        a.part[2 * blockIdx.x + 1] = bs[0];
    }
}

// one block of kMdBlocks threads: thermo row, uncertainty stop, step counter (or the invalid flag)
__global__ void __launch_bounds__(kMdBlocks) md_finish_kernel(MdArgs a) {
    __shared__ double ks[kMdBlocks], bs[kMdBlocks];
    if (md_frozen(a.state)) return;
    if (a.status[6] != 0) {
        if (threadIdx.x == 0) a.state[2] = 1;
        return;
    }
    ks[threadIdx.x] = a.part[2 * threadIdx.x];
    bs[threadIdx.x] = a.part[2 * threadIdx.x + 1];
    __syncthreads();
    for (int w = kMdBlocks / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            ks[threadIdx.x] += ks[threadIdx.x + w];
            bs[threadIdx.x] = nan_max(bs[threadIdx.x], bs[threadIdx.x + w]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        long long done = a.state[0];
        if (!a.init) {
            double* row = a.thermo + 11 * (done - a.state[3]);
            row[0] = a.ew_n[0];
            row[1] = ks[0];
            for (int k = 0; k < 9; ++k) row[2 + k] = a.ew_n[2 + k];
            a.state[0] = ++done;
        }
        if (a.stop_on_uncertain && bs[0] > a.ediff) a.state[1] = done;
    }
}

int md_check_args(sgpr_context* h, int64_t N, const double* cell_h, const int32_t* pbc_h, const sgpr_md_params* p,
                  const void* F_d, const double* beta_d, const int64_t* state_d) {
    if (!h || !cell_h || !pbc_h || !p || !F_d || !state_d) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    if (N < 0 || N > 0x7fffff00ll) {
        set_error("bad atom count");
        return SGPR_ERR_INVALID;
    }
    if (!isfinite(p->dt) || (p->langevin && (!(p->friction >= 0.0) || !isfinite(p->friction) || !(p->kT >= 0.0) || !isfinite(p->kT)))) {
        set_error("MD parameters: dt must be finite, friction and kT finite and >= 0");
        return SGPR_ERR_INVALID;
    }
    if (p->stop_on_uncertain && !beta_d) {
        set_error("stop_on_uncertain needs beta_d");
        return SGPR_ERR_INVALID;
    }
    SGPR_CUDA(cudaSetDevice(h->device));
    SGPR_TRY(h->md_pos.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    SGPR_TRY(h->md_mom.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    SGPR_TRY(h->md_F.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    SGPR_TRY(h->md_beta.ensure(sizeof(double) * ((size_t)N + 1)));
    SGPR_TRY(h->md_ew.ensure(sizeof(double) * 16));
    SGPR_TRY(h->md_part.ensure(sizeof(double) * 2 * kMdBlocks));
    return SGPR_OK;
}

MdArgs md_args(sgpr_context* h, int64_t N, double* pos_d, double* mom_d, const double* mass_d, const sgpr_md_params* p,
               double* F_d, double* thermo_d, double* beta_d, int64_t* state_d, bool init) {
    MdArgs a{};
    a.N = N;
    a.dt = p->dt;
    a.half_dt = 0.5 * p->dt;
    a.c1 = p->langevin ? exp(-p->friction * p->dt) : 1.0;
    a.c2 = p->langevin ? sqrt(1.0 - a.c1 * a.c1) : 0.0;
    a.kT = p->kT;
    a.ediff = p->ediff;
    a.seed = p->seed;
    a.langevin = p->langevin ? 1 : 0;
    a.stop_on_uncertain = p->stop_on_uncertain ? 1 : 0;
    a.init = init ? 1 : 0;
    a.pos = pos_d;
    a.mom = mom_d;
    a.mass = mass_d;
    a.F = F_d;
    a.beta = beta_d;
    a.pos_n = h->md_pos.as<double>();
    a.mom_n = h->md_mom.as<double>();
    a.F_n = h->md_F.as<double>();
    a.beta_n = h->md_beta.as<double>();
    a.ew_n = h->md_ew.as<double>();
    a.part = h->md_part.as<double>();
    a.thermo = thermo_d;
    a.state = reinterpret_cast<long long*>(state_d);
    a.status = h->status_d.as<long long>();
    return a;
}

int md_grid(int64_t N) { return (int)std::min<int64_t>(std::max<int64_t>((N + kMdThreads - 1) / kMdThreads, 1), 4096); }

// prediction of the step's positions + kick/commit + finish.  graph: the prediction may replay sgpr_predict's own
// graph (plain launches are needed while the caller captures the whole step)
int md_evaluate(sgpr_context* h, const MdArgs& a, const double* pos, const int32_t* Z_d, const double* cell_h,
                const int32_t* pbc_h, cudaStream_t st, bool graph) {
    double* ew = const_cast<double*>(a.ew_n);
    SGPR_TRY(md_predict(h, a.N, pos, Z_d, cell_h, pbc_h, st, ew, const_cast<double*>(a.F_n), ew + 2,
                        a.beta ? const_cast<double*>(a.beta_n) : nullptr, graph));
    // a sizing step validated itself on the host; status[6] may still hold the verdict of an earlier warm step
    if (!h->step_was_warm) SGPR_CUDA(cudaMemsetAsync(h->status_d.as<long long>() + 6, 0, sizeof(long long), st));
    md_kick_kernel<<<kMdBlocks, kMdThreads, 0, st>>>(a);
    md_finish_kernel<<<1, kMdBlocks, 0, st>>>(a);
    SGPR_CUDA(cudaGetLastError());
    return SGPR_OK;
}

int md_enqueue_step(sgpr_context* h, const MdArgs& a, const int32_t* Z_d, const double* cell_h, const int32_t* pbc_h,
                    cudaStream_t st, bool graph) {
    md_drift_kernel<<<md_grid(a.N), kMdThreads, 0, st>>>(a);
    SGPR_CUDA(cudaGetLastError());
    return md_evaluate(h, a, a.pos_n, Z_d, cell_h, pbc_h, st, graph);
}

int md_step(sgpr_context* h, const MdArgs& a, const int32_t* Z_d, const double* cell_h, const int32_t* pbc_h,
            cudaStream_t st, const sgpr_md_params* p) {
    sgpr_context::DriverGraphKey key;
    memset(&key, 0, sizeof(key));
    key.driver = kDriverMd;
    key.N = a.N;
    key.stream = (void*)st;
    key.ptr[0] = a.pos; key.ptr[1] = a.mom; key.ptr[2] = Z_d; key.ptr[3] = a.mass;
    key.ptr[4] = a.F; key.ptr[5] = a.thermo; key.ptr[6] = a.beta; key.ptr[7] = a.state;
    for (int i = 0; i < 9; ++i) key.cell[i] = cell_h[i];
    key.prm[0] = p->dt; key.prm[1] = a.c1; key.prm[2] = a.c2; key.prm[3] = a.kT; key.prm[4] = a.ediff;
    key.seed = a.seed;
    key.flag[0] = a.langevin;
    key.flag[1] = a.stop_on_uncertain;
    return driver_graph_step(h, key, md_warm_possible(h, a.N, pbc_h, a.beta != nullptr),
                             [&](bool graph) { return md_enqueue_step(h, a, Z_d, cell_h, pbc_h, st, graph); });
}

}  // namespace

int driver_name_step(sgpr_context* h, int rc, const long long* state_d, cudaStream_t st, const char* what) {
    char msg[768];
    snprintf(msg, sizeof(msg), "%s", sgpr_last_error());
    long long done = -1;
    if (cudaStreamSynchronize(st) == cudaSuccess && cudaMemcpy(&done, state_d, sizeof(done), cudaMemcpyDeviceToHost) == cudaSuccess)
        set_error("%s %lld: %s", what, done + 1, msg);
    else
        cudaGetLastError();
    h->warm_ok = false;
    return rc;
}

int driver_graph_step(sgpr_context* h, const sgpr_context::DriverGraphKey& key, bool warm,
                      const std::function<int(bool)>& enqueue) {
    if (!warm || !h->use_graph || h->timing) return enqueue(true);
    cudaStream_t st = (cudaStream_t)key.stream;
    // a workspace was reallocated since capture: the graphs point at freed memory
    const unsigned long long gen = buf_generation();
    if (gen != h->driver_graph_gen) {
        drop_driver_graphs(h);
        h->driver_graph_gen = gen;
    }
    for (auto& e : h->driver_graphs) {
        if (memcmp(&e.key, &key, sizeof(key)) == 0) {
            e.stamp = ++h->graph_clock;
            h->step_was_warm = true;
            SGPR_CUDA(cudaGraphLaunch(e.exec, st));
            return SGPR_OK;
        }
    }
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
        cudaGetLastError();   // e.g. the legacy default stream cannot be captured
        return enqueue(true);
    }
    const int rc = enqueue(false);
    const cudaError_t ce = cudaStreamEndCapture(st, &graph);
    if (rc != SGPR_OK || ce != cudaSuccess || !graph || !h->step_was_warm) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        h->use_graph = false;   // plain launches from now on (as predict_impl does)
        h->warm_ok = false;     // whatever was enqueued during the failed capture never ran
        if (rc != SGPR_OK) return rc;
        return enqueue(false);
    }
    cudaGraphExec_t exec = nullptr;
    if (buf_generation() != h->driver_graph_gen || cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
        // (a workspace grown during the capture would leave a graph that points at freed memory)
        cudaGraphDestroy(graph);
        cudaGetLastError();
        h->warm_ok = false;
        return enqueue(false);
    }
    cudaGraphDestroy(graph);
    if (h->driver_graphs.size() >= 4) {   // evict the least recently used entry
        size_t lru = 0;
        for (size_t i = 1; i < h->driver_graphs.size(); ++i)
            if (h->driver_graphs[i].stamp < h->driver_graphs[lru].stamp) lru = i;
        cudaGraphExecDestroy(h->driver_graphs[lru].exec);
        h->driver_graphs.erase(h->driver_graphs.begin() + lru);
    }
    sgpr_context::DriverGraphEntry e;
    e.key = key;
    e.exec = exec;
    e.stamp = ++h->graph_clock;
    h->driver_graphs.push_back(e);
    SGPR_CUDA(cudaGraphLaunch(exec, st));
    return SGPR_OK;
}

void drop_driver_graphs(sgpr_context* h) {
    for (auto& e : h->driver_graphs) cudaGraphExecDestroy(e.exec);
    h->driver_graphs.clear();
}

}  // namespace sgpr

using namespace sgpr;

extern "C" __attribute__((visibility("default"))) int sgpr_md_init(sgpr_handle h, int64_t N, const double* pos_d,
                                                                   const int32_t* Z_d, const double* cell_h,
                                                                   const int32_t* pbc_h, const sgpr_md_params* p,
                                                                   void* stream, double* F_d, double* beta_d,
                                                                   int64_t* state_d) {
    SGPR_TRY(md_check_args(h, N, cell_h, pbc_h, p, F_d, beta_d, state_d));
    cudaStream_t st = (cudaStream_t)stream;
    const MdArgs a = md_args(h, N, nullptr, nullptr, nullptr, p, F_d, nullptr, p->stop_on_uncertain ? beta_d : nullptr,
                             state_d, true);
    md_reset_kernel<<<1, 1, 0, st>>>(a.state);
    SGPR_CUDA(cudaGetLastError());
    return md_evaluate(h, a, pos_d, Z_d, cell_h, pbc_h, st, true);
}

extern "C" __attribute__((visibility("default"))) int sgpr_md_steps(sgpr_handle h, int64_t N, double* pos_d, double* mom_d,
                                                                    const int32_t* Z_d, const double* mass_d,
                                                                    const double* cell_h, const int32_t* pbc_h,
                                                                    const sgpr_md_params* p, int32_t n_steps, void* stream,
                                                                    double* F_d, double* thermo_d, double* beta_d,
                                                                    int64_t* state_d) {
    SGPR_TRY(md_check_args(h, N, cell_h, pbc_h, p, F_d, beta_d, state_d));
    if (n_steps < 0 || (n_steps > 0 && (!thermo_d || (N > 0 && (!pos_d || !mom_d || !mass_d || !Z_d))))) {
        set_error("null argument or n_steps < 0");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const MdArgs a = md_args(h, N, pos_d, mom_d, mass_d, p, F_d, thermo_d, p->stop_on_uncertain ? beta_d : nullptr,
                             state_d, false);
    md_begin_kernel<<<1, 1, 0, st>>>(a.state);
    SGPR_CUDA(cudaGetLastError());
    for (int32_t k = 0; k < n_steps; ++k) {
        const int rc = md_step(h, a, Z_d, cell_h, pbc_h, st, p);
        if (rc != SGPR_OK) return driver_name_step(h, rc, a.state, st, "MD step");
    }
    return SGPR_OK;
}
