// Geometry relaxation on the device (include/sgpr_b200.h: sgpr_relax_init, sgpr_relax_steps): ASE's FIRE around the
// prediction step, with positions, velocities and forces resident in HBM and no host synchronisation per step.
//
// A step is  move (FIRE branch, v, dr into scratch, |dr|^2 partials)  ->  place (|dr| in a fixed order, maxstep, the
// scratch positions)  ->  prediction of the scratch positions  ->  commit (r, v, F, beta; F of fixed atoms zeroed; F.v,
// F.F, v.v, max |F_i|^2, max beta partials)  ->  finish (trace row, FIRE scalars, converged / uncertain step, counter).
// As in md.cu nothing reaches pos/vel/F/beta/fire unless the prediction was valid, the counters live on the device and a
// warm step replays one CUDA graph.  The FIRE branch of step k is a function of what the finish of step k-1 left in
// fire_d and state_d: the move kernel evaluates it in every thread, the finish kernel commits it.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "sgpr_internal.cuh"

namespace sgpr {
namespace {

constexpr int kRxBlocks = 128;    // fixed grid of move / place / commit: partials are summed in a fixed order
constexpr int kRxThreads = 256;
constexpr int kRxParts = 5;       // commit partials per block: F.v, F.F, v.v, max |F_i|^2, max beta

struct RxArgs {
    long long N;
    double maxstep, dtmax, finc, fdec, astart, fa, fmax2, ediff;
    long long Nmin;
    int stop_on_uncertain, init;
    double* pos;
    double* vel;
    const unsigned char* fixed;   // nullptr: no fixed atoms
    double* F;
    double* beta;                 // nullptr: no covloss
    double* fire;                 // [6] dt, a, F.v, F.F, v.v, max |F_i|^2
    double* pos_n;                // scratch of the step in flight: dr (move), then the positions (place)
    double* vel_n;
    const double* F_n;
    const double* beta_n;
    const double* ew_n;           // [E, pad, W(9)]
    double* part;                 // [kRxBlocks][kRxParts] commit partials, then [kRxBlocks] |dr|^2 partials
    double* trace;                // [n_steps, 13]
    long long* state;             // {steps done, uncertain step, invalid, first step of the call, converged step, Nsteps}
    const long long* status;      // nl.cu status block: [6] = 1 when the prediction of this step was invalid
};

__device__ __forceinline__ bool rx_frozen(const long long* s) { return s[1] >= 0 || s[2] != 0 || s[4] >= 0; }

// FIRE's velocity rule and scalar update of the next step, from the committed state
struct FireStep {
    int mix;           // 1: v = (1-a_mix) v + a_mix |v| F/|F|;  0: v = 0 (first step) or v *= 0 (reset)
    int first;
    double a_mix, dt, a;
    long long nsteps;
};

__device__ __forceinline__ FireStep fire_step(const RxArgs& a) {
    FireStep f;
    f.dt = a.fire[0];
    f.a = a.fire[1];
    f.a_mix = f.a;
    f.nsteps = a.state[5];
    f.first = a.state[0] == 0;
    f.mix = 0;
    if (f.first) return f;
    if (a.fire[2] > 0.0) {
        f.mix = 1;
        if (f.nsteps > a.Nmin) {
            const double t = __dmul_rn(f.dt, a.finc);
            f.dt = a.dtmax < t ? a.dtmax : t;   // Python's min(t, dtmax)
            f.a = __dmul_rn(f.a, a.fa);
        }
        f.nsteps += 1;
    } else {
        f.a = a.astart;
        f.dt = __dmul_rn(f.dt, a.fdec);
        f.nsteps = 0;
    }
    return f;
}

template <int T>
__device__ __forceinline__ void block_sum(double* s) {
    __syncthreads();
    for (int w = T / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) s[threadIdx.x] += s[threadIdx.x + w];
        __syncthreads();
    }
}

__global__ void rx_reset_kernel(long long* state, double* fire, double dt, double a) {
    state[0] = 0;
    state[1] = -1;
    state[2] = 0;
    state[3] = 0;
    state[4] = -1;
    state[5] = 0;
    fire[0] = dt;
    fire[1] = a;
    for (int k = 2; k < 6; ++k) fire[k] = 0.0;
}

// ASE's run(fmax) tests the current forces before the first step of every call
__global__ void rx_begin_kernel(long long* state, const double* fire, double fmax2) {
    state[2] = 0;
    state[3] = state[0];
    state[4] = fire[5] < fmax2 ? state[0] : -1;
}

// v and dr of FIRE in the operation order of ase/optimize/fire.py (explicit roundings: no contraction into FMA)
__global__ void __launch_bounds__(kRxThreads) rx_move_kernel(RxArgs a) {
    __shared__ double ds[kRxThreads];
    if (rx_frozen(a.state)) return;
    const FireStep f = fire_step(a);
    const double nF = __dsqrt_rn(a.fire[3]), nv = __dsqrt_rn(a.fire[4]);
    const double keep = __dsub_rn(1.0, f.a_mix);
    double d2 = 0.0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.N; i += (long long)gridDim.x * blockDim.x) {
        for (int c = 0; c < 3; ++c) {
            const double F = a.F[3 * i + c];
            double v = f.first ? 0.0 : a.vel[3 * i + c];
            if (f.mix)
                v = __dadd_rn(__dmul_rn(keep, v), __dmul_rn(__ddiv_rn(__dmul_rn(f.a_mix, F), nF), nv));
            else
                v = __dmul_rn(v, 0.0);
            v = __dadd_rn(v, __dmul_rn(f.dt, F));
            const double dr = __dmul_rn(f.dt, v);
            a.vel_n[3 * i + c] = v;
            a.pos_n[3 * i + c] = dr;
            d2 += dr * dr;
        }
    }
    ds[threadIdx.x] = d2;
    block_sum<kRxThreads>(ds);
    if (threadIdx.x == 0) a.part[kRxParts * kRxBlocks + blockIdx.x] = ds[0];
}

// every block sums the |dr|^2 partials in the same order, then r_n = r + dr (scaled to maxstep)
__global__ void __launch_bounds__(kRxThreads) rx_place_kernel(RxArgs a) {
    __shared__ double ds[kRxBlocks];
    if (rx_frozen(a.state)) return;
    if (threadIdx.x < kRxBlocks) ds[threadIdx.x] = a.part[kRxParts * kRxBlocks + threadIdx.x];
    block_sum<kRxBlocks>(ds);
    const double norm = __dsqrt_rn(ds[0]);
    const bool scale = norm > a.maxstep;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.N; i += (long long)gridDim.x * blockDim.x) {
        for (int c = 0; c < 3; ++c) {
            double dr = a.pos_n[3 * i + c];
            if (scale) dr = __ddiv_rn(__dmul_rn(a.maxstep, dr), norm);
            a.pos_n[3 * i + c] = __dadd_rn(a.pos[3 * i + c], dr);
        }
    }
}

// commit of a valid step (init: of the starting forces only); per-block F.v, F.F, v.v, max |F_i|^2, max beta
__global__ void __launch_bounds__(kRxThreads) rx_commit_kernel(RxArgs a) {
    __shared__ double fv[kRxThreads], ff[kRxThreads], vv[kRxThreads], fm[kRxThreads], bm[kRxThreads];
    if (rx_frozen(a.state) || a.status[6] != 0) return;
    double s_fv = 0.0, s_ff = 0.0, s_vv = 0.0, fmax2 = -INFINITY, bmax = -INFINITY;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.N; i += (long long)gridDim.x * blockDim.x) {
        const bool fixed = a.fixed && a.fixed[i];
        double f[3];
        for (int c = 0; c < 3; ++c) {
            f[c] = fixed ? 0.0 : a.F_n[3 * i + c];
            a.F[3 * i + c] = f[c];
            s_ff += f[c] * f[c];
            if (!a.init) {
                const double v = a.vel_n[3 * i + c];
                a.vel[3 * i + c] = v;
                a.pos[3 * i + c] = a.pos_n[3 * i + c];
                s_fv += f[c] * v;
                s_vv += v * v;
            }
        }
        // (F**2).sum(axis=1) of numpy
        fmax2 = nan_max(fmax2, __dadd_rn(__dadd_rn(__dmul_rn(f[0], f[0]), __dmul_rn(f[1], f[1])), __dmul_rn(f[2], f[2])));
        if (a.beta) {
            const double b = a.beta_n[i];
            a.beta[i] = b;
            bmax = nan_max(bmax, b);
        }
    }
    fv[threadIdx.x] = s_fv;
    ff[threadIdx.x] = s_ff;
    vv[threadIdx.x] = s_vv;
    fm[threadIdx.x] = fmax2;
    bm[threadIdx.x] = bmax;
    __syncthreads();
    for (int w = kRxThreads / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            fv[threadIdx.x] += fv[threadIdx.x + w];
            ff[threadIdx.x] += ff[threadIdx.x + w];
            vv[threadIdx.x] += vv[threadIdx.x + w];
            fm[threadIdx.x] = nan_max(fm[threadIdx.x], fm[threadIdx.x + w]);
            bm[threadIdx.x] = nan_max(bm[threadIdx.x], bm[threadIdx.x + w]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double* p = a.part + kRxParts * blockIdx.x;
        p[0] = fv[0];
        p[1] = ff[0];
        p[2] = vv[0];
        p[3] = fm[0];
        p[4] = bm[0];
    }
}

// one block of kRxBlocks threads: FIRE scalars of the step, trace row, reductions of the committed F and v, converged
// and uncertain step, step counter (or the invalid flag)
__global__ void __launch_bounds__(kRxBlocks) rx_finish_kernel(RxArgs a) {
    __shared__ double fv[kRxBlocks], ff[kRxBlocks], vv[kRxBlocks], fm[kRxBlocks], bm[kRxBlocks];
    if (rx_frozen(a.state)) return;
    if (a.status[6] != 0) {
        if (threadIdx.x == 0) a.state[2] = 1;
        return;
    }
    const double* p = a.part + kRxParts * threadIdx.x;
    fv[threadIdx.x] = p[0];
    ff[threadIdx.x] = p[1];
    vv[threadIdx.x] = p[2];
    fm[threadIdx.x] = p[3];
    bm[threadIdx.x] = p[4];
    __syncthreads();
    for (int w = kRxBlocks / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            fv[threadIdx.x] += fv[threadIdx.x + w];
            ff[threadIdx.x] += ff[threadIdx.x + w];
            vv[threadIdx.x] += vv[threadIdx.x + w];
            fm[threadIdx.x] = nan_max(fm[threadIdx.x], fm[threadIdx.x + w]);
            bm[threadIdx.x] = nan_max(bm[threadIdx.x], bm[threadIdx.x + w]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        long long done = a.state[0];
        if (!a.init) {
            const FireStep f = fire_step(a);
            a.fire[0] = f.dt;
            a.fire[1] = f.a;
            a.state[5] = f.nsteps;
            double* row = a.trace + 13 * (done - a.state[3]);
            row[0] = a.ew_n[0];
            row[1] = sqrt(fm[0]);
            row[2] = f.dt;
            row[3] = f.a;
            for (int k = 0; k < 9; ++k) row[4 + k] = a.ew_n[2 + k];
            a.state[0] = ++done;
            a.fire[2] = fv[0];
            a.fire[4] = vv[0];
        }
        a.fire[3] = ff[0];
        a.fire[5] = fm[0];
        if (a.stop_on_uncertain && bm[0] > a.ediff) a.state[1] = done;
        if (fm[0] < a.fmax2) a.state[4] = done;
    }
}

int rx_check_args(sgpr_context* h, int64_t N, const double* cell_h, const int32_t* pbc_h, const sgpr_relax_params* p,
                  const void* F_d, const double* beta_d, const double* fire_d, const int64_t* state_d) {
    if (!h || !cell_h || !pbc_h || !p || !F_d || !fire_d || !state_d) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    if (N < 0 || N > 0x7fffff00ll) {
        set_error("bad atom count");
        return SGPR_ERR_INVALID;
    }
    const double pos[] = {p->dt, p->maxstep, p->dtmax, p->finc, p->fdec};
    bool ok = isfinite(p->astart) && isfinite(p->fa) && isfinite(p->a) && isfinite(p->fmax) && p->fmax >= 0.0 && p->Nmin >= 0;
    for (double x : pos) ok = ok && isfinite(x) && x > 0.0;
    if (!ok) {
        set_error("FIRE parameters: dt, maxstep, dtmax, finc, fdec must be finite and > 0, astart, fa, a finite, "
                  "fmax finite and >= 0, Nmin >= 0");
        return SGPR_ERR_INVALID;
    }
    if (p->stop_on_uncertain && !beta_d) {
        set_error("stop_on_uncertain needs beta_d");
        return SGPR_ERR_INVALID;
    }
    SGPR_CUDA(cudaSetDevice(h->device));
    SGPR_TRY(h->rx_pos.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    SGPR_TRY(h->rx_vel.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    SGPR_TRY(h->rx_F.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    SGPR_TRY(h->rx_beta.ensure(sizeof(double) * ((size_t)N + 1)));
    SGPR_TRY(h->rx_ew.ensure(sizeof(double) * 16));
    SGPR_TRY(h->rx_part.ensure(sizeof(double) * (kRxParts + 1) * kRxBlocks));
    return SGPR_OK;
}

RxArgs rx_args(sgpr_context* h, int64_t N, double* pos_d, double* vel_d, const uint8_t* fixed_d,
               const sgpr_relax_params* p, double* F_d, double* trace_d, double* beta_d, double* fire_d,
               int64_t* state_d, bool init) {
    RxArgs a{};
    a.N = N;
    a.maxstep = p->maxstep;
    a.dtmax = p->dtmax;
    a.finc = p->finc;
    a.fdec = p->fdec;
    a.astart = p->astart;
    a.fa = p->fa;
    a.fmax2 = p->fmax * p->fmax;
    a.ediff = p->ediff;
    a.Nmin = p->Nmin;
    a.stop_on_uncertain = p->stop_on_uncertain ? 1 : 0;
    a.init = init ? 1 : 0;
    a.pos = pos_d;
    a.vel = vel_d;
    a.fixed = fixed_d;
    a.F = F_d;
    a.beta = beta_d;
    a.fire = fire_d;
    a.pos_n = h->rx_pos.as<double>();
    a.vel_n = h->rx_vel.as<double>();
    a.F_n = h->rx_F.as<double>();
    a.beta_n = h->rx_beta.as<double>();
    a.ew_n = h->rx_ew.as<double>();
    a.part = h->rx_part.as<double>();
    a.trace = trace_d;
    a.state = reinterpret_cast<long long*>(state_d);
    a.status = h->status_d.as<long long>();
    return a;
}

// prediction of the step's positions + commit + finish (graph: as md.cu's md_evaluate)
int rx_evaluate(sgpr_context* h, const RxArgs& a, const double* pos, const int32_t* Z_d, const double* cell_h,
                const int32_t* pbc_h, cudaStream_t st, bool graph) {
    double* ew = const_cast<double*>(a.ew_n);
    SGPR_TRY(md_predict(h, a.N, pos, Z_d, cell_h, pbc_h, st, ew, const_cast<double*>(a.F_n), ew + 2,
                        a.beta ? const_cast<double*>(a.beta_n) : nullptr, graph));
    // a sizing step validated itself on the host; status[6] may still hold the verdict of an earlier warm step
    if (!h->step_was_warm) SGPR_CUDA(cudaMemsetAsync(h->status_d.as<long long>() + 6, 0, sizeof(long long), st));
    rx_commit_kernel<<<kRxBlocks, kRxThreads, 0, st>>>(a);
    rx_finish_kernel<<<1, kRxBlocks, 0, st>>>(a);
    SGPR_CUDA(cudaGetLastError());
    return SGPR_OK;
}

int rx_enqueue_step(sgpr_context* h, const RxArgs& a, const int32_t* Z_d, const double* cell_h, const int32_t* pbc_h,
                    cudaStream_t st, bool graph) {
    rx_move_kernel<<<kRxBlocks, kRxThreads, 0, st>>>(a);
    rx_place_kernel<<<kRxBlocks, kRxThreads, 0, st>>>(a);
    SGPR_CUDA(cudaGetLastError());
    return rx_evaluate(h, a, a.pos_n, Z_d, cell_h, pbc_h, st, graph);
}

int rx_step(sgpr_context* h, const RxArgs& a, const int32_t* Z_d, const double* cell_h, const int32_t* pbc_h,
            cudaStream_t st, const sgpr_relax_params* p) {
    sgpr_context::DriverGraphKey key;
    memset(&key, 0, sizeof(key));
    key.driver = kDriverRelax;
    key.N = a.N;
    key.stream = (void*)st;
    key.ptr[0] = a.pos; key.ptr[1] = a.vel; key.ptr[2] = Z_d; key.ptr[3] = a.fixed; key.ptr[4] = a.F;
    key.ptr[5] = a.trace; key.ptr[6] = a.beta; key.ptr[7] = a.state; key.ptr[8] = a.fire;
    for (int i = 0; i < 9; ++i) key.cell[i] = cell_h[i];
    key.prm[0] = p->maxstep; key.prm[1] = p->dtmax; key.prm[2] = p->finc; key.prm[3] = p->fdec;
    key.prm[4] = p->astart; key.prm[5] = p->fa; key.prm[6] = a.fmax2; key.prm[7] = a.ediff;
    key.seed = (uint64_t)a.Nmin;
    key.flag[0] = a.stop_on_uncertain;
    return driver_graph_step(h, key, md_warm_possible(h, a.N, pbc_h, a.beta != nullptr),
                             [&](bool graph) { return rx_enqueue_step(h, a, Z_d, cell_h, pbc_h, st, graph); });
}

}  // namespace
}  // namespace sgpr

using namespace sgpr;

extern "C" __attribute__((visibility("default"))) int sgpr_relax_init(sgpr_handle h, int64_t N, const double* pos_d,
                                                                      const int32_t* Z_d, const uint8_t* fixed_d,
                                                                      const double* cell_h, const int32_t* pbc_h,
                                                                      const sgpr_relax_params* p, void* stream,
                                                                      double* F_d, double* beta_d, double* fire_d,
                                                                      int64_t* state_d) {
    SGPR_TRY(rx_check_args(h, N, cell_h, pbc_h, p, F_d, beta_d, fire_d, state_d));
    cudaStream_t st = (cudaStream_t)stream;
    const RxArgs a = rx_args(h, N, nullptr, nullptr, fixed_d, p, F_d, nullptr, p->stop_on_uncertain ? beta_d : nullptr,
                             fire_d, state_d, true);
    rx_reset_kernel<<<1, 1, 0, st>>>(a.state, a.fire, p->dt, p->a);
    SGPR_CUDA(cudaGetLastError());
    return rx_evaluate(h, a, pos_d, Z_d, cell_h, pbc_h, st, true);
}

extern "C" __attribute__((visibility("default"))) int sgpr_relax_steps(sgpr_handle h, int64_t N, double* pos_d,
                                                                       double* vel_d, const int32_t* Z_d,
                                                                       const uint8_t* fixed_d, const double* cell_h,
                                                                       const int32_t* pbc_h, const sgpr_relax_params* p,
                                                                       int32_t n_steps, void* stream, double* F_d,
                                                                       double* trace_d, double* beta_d, double* fire_d,
                                                                       int64_t* state_d) {
    SGPR_TRY(rx_check_args(h, N, cell_h, pbc_h, p, F_d, beta_d, fire_d, state_d));
    if (n_steps < 0 || (n_steps > 0 && (!trace_d || (N > 0 && (!pos_d || !vel_d || !Z_d))))) {
        set_error("null argument or n_steps < 0");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const RxArgs a = rx_args(h, N, pos_d, vel_d, fixed_d, p, F_d, trace_d, p->stop_on_uncertain ? beta_d : nullptr,
                             fire_d, state_d, false);
    rx_begin_kernel<<<1, 1, 0, st>>>(a.state, a.fire, a.fmax2);
    SGPR_CUDA(cudaGetLastError());
    for (int32_t k = 0; k < n_steps; ++k) {
        const int rc = rx_step(h, a, Z_d, cell_h, pbc_h, st, p);
        if (rc != SGPR_OK) return driver_name_step(h, rc, a.state, st, "relaxation step");
    }
    return SGPR_OK;
}
