// C-ABI entry points of libsgpr_b200.so (include/sgpr_b200.h) and the per-step pipeline.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <cmath>

#include <nvtx3/nvToolsExt.h>

#include "sgpr_internal.cuh"

namespace sgpr {

// NVTX ranges on the reference's timing nodes (calculator/active.py:427-535: nl+desc | kernel | results | active):
// here nl / desc / gemm / force / covloss, visible in Nsight Systems / Compute next to the kernels they enclose.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

static thread_local char g_err[1024] = "";

static std::atomic<unsigned long long> g_buf_generation{0};
unsigned long long buf_generation() { return g_buf_generation.load(); }

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int DevBuf::ensure(size_t need) {
    if (need <= bytes) return SGPR_OK;
    if (p) cudaFree(p);
    p = nullptr;
    g_buf_generation.fetch_add(1);
    size_t want = need + need / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        bytes = 0;
        p = nullptr;
        set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        return SGPR_ERR_NOMEM;
    }
    bytes = want;
    return SGPR_OK;
}
void DevBuf::release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
}

// ---------------------------------------------------------------------------------
// small kernels of the pipeline
// ---------------------------------------------------------------------------------
__global__ void transpose_zhat_kernel(int D, int ldp, int m0, int Ms, int ld_zt, const double* __restrict__ zhat,
                                      double* __restrict__ zt) {
    // zt[e][m] = zhat[m0+m][e]
    __shared__ double tile[32][33];
    const int e0 = blockIdx.x * 32, mm0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int m = mm0 + r, e = e0 + threadIdx.x;
        tile[r][threadIdx.x] = (m < Ms && e < D) ? zhat[(size_t)(m0 + m) * ldp + e] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int e = e0 + r, m = mm0 + threadIdx.x;
        if (e < D && m < ld_zt) zt[(size_t)e * ld_zt + m] = tile[threadIdx.x][r];
    }
}

// per-atom terms outside the GEMM: constant mean (gppotential.py:219-227), the
// "lone atoms" kernel term (similarity.py:94-103), scatter of forces to caller order
__global__ void atom_terms_kernel(int64_t N, int n_active, const int* __restrict__ active,
                                  const AtomRec* __restrict__ atoms, const long long* __restrict__ nl_first,
                                  const unsigned char* __restrict__ owned, const double* __restrict__ mean_w,
                                  const double* __restrict__ lone_mu, double* __restrict__ part) {
    __shared__ double red[256];
    double s = 0.0;
    for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < n_active; env += gridDim.x * blockDim.x) {
        const int c = active ? active[env] : env;
        if (owned && !owned[c]) continue;
        const int sp = meta_species(atoms[c].meta);
        s += mean_w[sp];
        if (nl_first[env + 1] == nl_first[env]) s += lone_mu[sp];
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) part[blockIdx.x] = red[0];
}

// covloss (calculator/active.py:781-804): beta_i = sqrt(clamp(1 - c_i, 0)) * sqrt(vscale[Z_i])
__global__ void beta_finish_kernel(int n_active, const int* __restrict__ active, const AtomRec* __restrict__ atoms,
                                   const int* __restrict__ rowof, const long long* __restrict__ nl_first,
                                   const unsigned char* __restrict__ owned, const unsigned char* __restrict__ sp_on,
                                   const int* __restrict__ sp_enabled, const double* __restrict__ cpart, int n_part,
                                   int part_ld, const double* __restrict__ clone, const double* __restrict__ vscale,
                                   const double* __restrict__ prow, int normalized, double xi, double* __restrict__ beta) {
    for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < n_active; env += gridDim.x * blockDim.x) {
        const int c = active ? active[env] : env;
        if (owned && !owned[c]) continue;
        const unsigned long long meta = atoms[c].meta;
        const int sp = meta_species(meta);
        double cc = 0.0;
        const bool lone = nl_first[env + 1] == nl_first[env];
        if (lone) {
            cc = clone[sp];
        } else if (sp_on[sp]) {
            const int row = rowof[c];
            for (int p = 0; p < n_part; ++p) cc += cpart[(size_t)p * part_ld + row];
            // un-normalised descriptors: c / alpha with the self kernel alpha = k(x,x) = (p.p)^xi (active.py:784-791)
            if (!normalized) cc /= pow(prow[row] * prow[row], xi);
        }
        double b = sqrt(fmax(1.0 - cc, 0.0));
        // the reference divides c by the self kernel k(x,x) = 0 for an excluded centre -> NaN (active.py:784-791)
        if (!lone && !sp_enabled[sp]) b = nan("");
        beta[meta_orig(meta)] = b * sqrt(vscale[sp]);
    }
}

// local energies e_r = sum of the per-(column tile, warp) partials written by the kernel-matrix
// GEMM (fixed order -> reproducible); also block partial sums of the owned rows for the total.
struct RowSpecies {
    int n_part[SGPR_MAX_SPECIES];   // 0 where the species has no usable inducing points
    int S;
};
__global__ void row_energy_kernel(int n_rows, RowSpecies rs, const int* __restrict__ row_first,
                                  const double* __restrict__ part, int part_ld,
                                  const unsigned char* __restrict__ row_owned, double* __restrict__ erow,
                                  double* __restrict__ epart) {
    __shared__ double red[256];
    __shared__ int rf[SGPR_MAX_SPECIES + 1];
    if (threadIdx.x <= rs.S) rf[threadIdx.x] = row_first[threadIdx.x];   // species row ranges live on the device
    __syncthreads();
    double tot = 0.0;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += gridDim.x * blockDim.x) {
        int np = 0;
#pragma unroll
        for (int s = 0; s < SGPR_MAX_SPECIES; ++s)
            if (s < rs.S && r >= rf[s] && r < rf[s + 1]) np = rs.n_part[s];
        double e = 0.0;
        for (int p = 0; p < np; ++p) e += part[(size_t)p * part_ld + r];
        erow[r] = e;
        if (!row_owned || row_owned[r]) tot += e;
    }
    red[threadIdx.x] = tot;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) epart[blockIdx.x] = red[0];
}

__global__ void scatter_forces_kernel(int64_t N, const AtomRec* __restrict__ atoms, const double* __restrict__ fcell,
                                      const unsigned char* __restrict__ owned, double* __restrict__ F,
                                      unsigned char* __restrict__ owned_out, const long long* __restrict__ parity_src = nullptr,
                                      long long parity_stride = 0) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= N) return;
    // fused exchange step: the buffer of the step that has just been published (counter already advanced)
    if (parity_src && (((*parity_src) - 1) & 1)) fcell += parity_stride;
    const int i = meta_orig(atoms[c].meta);
    // atoms of other ranks: zero (the peer-memory exchange leaves what was pushed to their owners in this buffer)
    const bool mine = owned ? owned[c] != 0 : true;
    F[3 * (size_t)i] = mine ? fcell[3 * c] : 0.0;
    F[3 * (size_t)i + 1] = mine ? fcell[3 * c + 1] : 0.0;
    F[3 * (size_t)i + 2] = mine ? fcell[3 * c + 2] : 0.0;
    if (owned_out) owned_out[i] = mine ? 1 : 0;
}

// dL/dx = -F in the caller's order, plus per-block partials of sum_k x_k (x) F_k (for dL/dcell)
__global__ void vjp_finish_kernel(int64_t N, const AtomRec* __restrict__ atoms, const double* __restrict__ fcell,
                                  double* __restrict__ gpos, double* __restrict__ xf_part) {
    __shared__ double red[9][128];
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < N; c += (int64_t)gridDim.x * blockDim.x) {
        const AtomRec a = atoms[c];
        const int i = meta_orig(a.meta);
        const double f[3] = {fcell[3 * c], fcell[3 * c + 1], fcell[3 * c + 2]};
        const double x[3] = {a.x, a.y, a.z};
        for (int q = 0; q < 3; ++q) gpos[3 * (size_t)i + q] = -f[q];
        for (int p = 0; p < 3; ++p)
            for (int q = 0; q < 3; ++q) acc[p * 3 + q] += x[p] * f[q];
    }
    for (int q = 0; q < 9; ++q) red[q][threadIdx.x] = acc[q];
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o)
            for (int q = 0; q < 9; ++q) red[q][threadIdx.x] += red[q][threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x < 9) xf_part[blockIdx.x * 9 + threadIdx.x] = red[threadIdx.x][0];
}

__global__ void final_reduce_kernel(int n_e, const double* __restrict__ epart, int n_x, const double* __restrict__ xpart,
                                    int n_w, const double* __restrict__ wpart, double* __restrict__ E,
                                    double* __restrict__ W) {
    // one block of 10 warps, fixed summation order -> run-to-run reproducible E and W:
    // warp 0 sums the energy partials, warps 1..9 one virial component each (lane-strided partial sums, then a
    // fixed shuffle tree); all ten sums run concurrently
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double s = 0.0;
    if (warp == 0) {
        for (int i = lane; i < n_e; i += 32) s += epart[i];
        for (int i = lane; i < n_x; i += 32) s += xpart[i];
    } else if (warp < 10) {
        // batches of 8 independent loads per lane (the additions stay in a fixed order): the loop is bound by the
        // number of dependent L2 round trips, not by the 21 k values it reads
        const int q = warp - 1;
        for (int base = lane; base < n_w; base += 32 * 8) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = base + 32 * u;
                v[u] = i < n_w ? wpart[(size_t)i * 9 + q] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) s += v[u];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
        if (warp == 0)
            E[0] = s;
        else if (warp < 10)
            W[warp - 1] = s;
    }
}

__global__ void row_to_orig_kernel(int64_t N, const AtomRec* __restrict__ atoms, const int* __restrict__ rowof,
                                   int* __restrict__ orig_of_row) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= N) return;
    orig_of_row[rowof[c]] = meta_orig(atoms[c].meta);
}
__global__ void orig_to_row_kernel(int64_t N, const AtomRec* __restrict__ atoms, const int* __restrict__ rowof,
                                   int* __restrict__ row_of_orig) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= N) return;
    row_of_orig[meta_orig(atoms[c].meta)] = rowof[c];
}

__global__ void lone_k_kernel(int n_active, const int* __restrict__ active, const AtomRec* __restrict__ atoms,
                              const long long* __restrict__ nl_first, int M, const int* __restrict__ ind_sp,
                              const unsigned char* __restrict__ ind_lone, double* __restrict__ K, double lone_w) {
    // K[i,m] += 1 when both LCEs have no neighbours and the same species (similarity.py:94-103)
    for (int env = blockIdx.x; env < n_active; env += gridDim.x) {
        if (nl_first[env + 1] != nl_first[env]) continue;
        const int c = active ? active[env] : env;
        const int sp = meta_species(atoms[c].meta);
        const int i = meta_orig(atoms[c].meta);
        for (int m = threadIdx.x; m < M; m += blockDim.x)
            if (ind_lone[m] && ind_sp[m] == sp) K[(size_t)i * M + m] += lone_w;
    }
}

// Explicit environments against the inducing set: K[e, m] = [same species, centre enabled] (p_e . z_m)^xi
// (+ lone_w when both are neighbour-less), m in the caller's inducing order.  One block per environment.
__global__ void env_kernel_rows_kernel(int n_env, int M, int D, int ldp, const double* __restrict__ penv,
                                       const double* __restrict__ zhat, const int* __restrict__ env_sp,
                                       const unsigned char* __restrict__ env_lone, const int* __restrict__ perm,
                                       const int* __restrict__ ind_sp_sorted, const unsigned char* __restrict__ ind_lone_sorted,
                                       const int* __restrict__ sp_enabled, double xi, int xi_int, double lone_w,
                                       double* __restrict__ K) {
    const int e = blockIdx.x;
    if (e >= n_env) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const double* q = penv + (size_t)e * ldp;
    const int sp = env_sp[e];
    for (int p = warp; p < M; p += nwarps) {
        double k = 0.0;
        if (ind_sp_sorted[p] == sp) {
            if (env_lone[e] || ind_lone_sorted[p]) {
                k = (env_lone[e] && ind_lone_sorted[p]) ? lone_w : 0.0;
            } else if (sp_enabled[sp]) {
                const double* z = zhat + (size_t)p * ldp;
                double d = 0.0;
                for (int t = lane; t < D; t += 32) d = fma(q[t], z[t], d);
                for (int o = 16; o; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
                if (xi_int >= 1) {
                    k = d;
                    for (int t = 1; t < xi_int; ++t) k *= d;
                } else {
                    k = pow(d, xi);
                }
            }
        }
        if (lane == 0) K[(size_t)e * M + perm[p]] = k;
    }
}

// ---------------------------------------------------------------------------------
// exchange step of the atom-sharded path without NCCL: E + 3x3 virial travel through peer-mapped mailboxes, a stamped
// flag per (rank, step parity) doubles as the barrier after which a rank may read the forces its peers added to it
// ---------------------------------------------------------------------------------
// mailbox block of one rank: [2 parities][world slots][16 doubles]; slot r = {E, W[9], -, ..., stamp (int64 at [15])}
__global__ void p2p_zero_next_kernel(double* __restrict__ own_base, long long stride, long long n,
                                     const long long* __restrict__ step_counter) {
    // the accumulation buffer of the NEXT step (the one this step does not use)
    double* dst = own_base + ((((*step_counter) & 1) == 0) ? stride : 0);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dst[i] = 0.0;
}
// Halo forces of the atom-sharded path: what this rank accumulated for atoms it does not own goes to the owners'
// buffers (peer-mapped), coalesced over the cell order -- adjacent x-slabs are contiguous index ranges.
__global__ void p2p_push_kernel(long long n3, PeerForces peers, int rank) {
    const long long off = (peers.parity_src && ((*peers.parity_src) & 1)) ? peers.parity_stride : 0;
    const double* mine = peers.peer_f[rank] + off;
    const long long lo = 3ll * peers.bounds[rank], hi = 3ll * peers.bounds[rank + 1];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n3; i += (long long)gridDim.x * blockDim.x) {
        if (i >= lo && i < hi) continue;
        const double v = mine[i];
        if (v == 0.0) continue;
        const int j = (int)(i / 3);
        int r = 0;
#pragma unroll
        for (int q = 1; q < SGPR_MAX_RANKS; ++q)
            if (q < peers.world && j >= peers.bounds[q]) r = q;
        atomicAdd(peers.peer_f[r] + off + i, v);
    }
}
// One block: publish this rank's E + virial (and the step's stamp) to every peer's mailbox, then wait for every peer's
// stamp and reduce in rank order.  The step counter advances in between (scatter_forces_kernel reads it afterwards).
__global__ void p2p_publish_wait_kernel(int rank, int world, P2PPeers peers, const double* __restrict__ ew_local,
                                        long long* __restrict__ step_counter, double* __restrict__ E, double* __restrict__ W,
                                        long long* __restrict__ status) {
    __shared__ double acc[SGPR_MAX_RANKS][10];
    __shared__ int timed_out;
    // every earlier kernel of this stream (the force kernel, the halo push with its remote red.add) has completed
    const long long stamp = *step_counter + 1;
    const int parity = (int)((stamp - 1) & 1);
    const int r = threadIdx.x;
    if (r == 0) timed_out = 0;
    if (r < world) {
        double* slot = peers.mail[r] + ((size_t)parity * world + rank) * 16;
        for (int q = 0; q < 10; ++q) slot[q] = ew_local[q];
        __threadfence_system();
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(reinterpret_cast<unsigned long long*>(slot + 15)),
                     "l"((unsigned long long)stamp)
                     : "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) *step_counter = stamp;
    if (r < world) {
        const double* slot = peers.mail[rank] + ((size_t)parity * world + r) * 16;
        unsigned long long t0, t1, seen = 0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(reinterpret_cast<const unsigned long long*>(slot + 15)) : "memory");
            if ((long long)seen >= stamp) break;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 10000000000ull) {   // 10 s: a peer died; never hang the GPU
                timed_out = 1;
                break;
            }
            __nanosleep(200);
        }
        for (int q = 0; q < 10; ++q) acc[r][q] = slot[q];
    }
    __syncthreads();
    if (threadIdx.x < 10) {
        double v = 0.0;
        for (int k = 0; k < world; ++k) v += acc[k][threadIdx.x];   // fixed order: every rank gets the same bits
        if (threadIdx.x == 0)
            E[0] = v;
        else
            W[threadIdx.x - 1] = v;
    }
    if (threadIdx.x == 0 && timed_out) {
        status[1] += 1;
        status[2] = 3;
    }
}

// CSR neighbour list in the caller's atom order (parity hook)
__global__ void nl_count_orig_kernel(int64_t N, const AtomRec* __restrict__ atoms, const long long* __restrict__ nl_first,
                                     long long* __restrict__ cnt) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c > N) return;
    if (c == N) {
        cnt[N] = 0;
        return;
    }
    cnt[meta_orig(atoms[c].meta)] = nl_first[c + 1] - nl_first[c];
}
__global__ void nl_export_kernel(int64_t N, const AtomRec* __restrict__ atoms, const PairRec* __restrict__ pairs,
                                 const long long* __restrict__ nl_first, const long long* __restrict__ first_out,
                                 int32_t* __restrict__ j_out, int8_t* __restrict__ S_out) {
    const int lane = threadIdx.x & 31;
    const int64_t c = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (c >= N) return;
    const AtomRec ai = atoms[c];
    const long long o = first_out[meta_orig(ai.meta)];
    const long long beg = nl_first[c], end = nl_first[c + 1];
    for (long long k = beg + lane; k < end; k += 32) {
        const PairRec pr = pairs[k];
        const AtomRec aj = atoms[pr.j];
        j_out[o + (k - beg)] = meta_orig(aj.meta);
        for (int q = 0; q < 3; ++q)
            S_out[3 * (o + (k - beg)) + q] = (int8_t)(pr.sb[q] - meta_w(aj.meta, q) + meta_w(ai.meta, q));
    }
}

// Per-structure sums of a batch, one warp per structure: E = local energies + mean + lone-atom terms
// (atom_terms_kernel's work), W = the environments' virials.  A structure is the cell-order range first[b] ..
// first[b+1]-1 (structure-major keys), whose order depends on that structure alone; lane-strided partial sums and a
// fixed shuffle tree make E and W reproducible and independent of the rest of the batch.
__global__ void batch_reduce_kernel(int B, const long long* __restrict__ first, const AtomRec* __restrict__ atoms,
                                    const int* __restrict__ rowof, const long long* __restrict__ nl_first,
                                    const double* __restrict__ erow, const double* __restrict__ mean_w,
                                    const double* __restrict__ lone_mu, const double* __restrict__ wenv,
                                    double* __restrict__ E, double* __restrict__ W) {
    const int lane = threadIdx.x & 31;
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    double e = 0.0, w[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (long long c = first[b] + lane; c < first[b + 1]; c += 32) {
        const int sp = meta_species(atoms[c].meta);
        e += erow[rowof[c]];
        e += mean_w[sp];
        if (nl_first[c + 1] == nl_first[c]) e += lone_mu[sp];
#pragma unroll
        for (int q = 0; q < 9; ++q) w[q] += wenv[9 * c + q];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        e += __shfl_xor_sync(0xffffffffu, e, o);
#pragma unroll
        for (int q = 0; q < 9; ++q) w[q] += __shfl_xor_sync(0xffffffffu, w[q], o);
    }
    if (lane == 0) {
        E[b] = e;
#pragma unroll
        for (int q = 0; q < 9; ++q) W[9 * (size_t)b + q] = w[q];
    }
}

// Ke[b, col] = sum over the atoms of structure b of K[i, m0 + col] (caller's order, lone-lone term included), one thread
// per (structure, column), atoms in order: a structure's sums do not depend on the rest of the batch.
__global__ void ke_reduce_kernel(int B, const long long* __restrict__ first, int M, int m0, int ncol,
                                 const double* __restrict__ K, double* __restrict__ Ke) {
    const long long n = (long long)B * ncol;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / ncol), col = (int)(t - (long long)b * ncol);
        double s = 0.0;
        for (long long i = first[b]; i < first[b + 1]; ++i) s += K[i * M + m0 + col];
        Ke[t] = s;
    }
}

}  // namespace sgpr

using namespace sgpr;

// =====================================================================================
// life cycle
// =====================================================================================
extern "C" __attribute__((visibility("default"))) const char* sgpr_last_error(void) { return g_err; }
extern "C" __attribute__((visibility("default"))) int sgpr_abi_version(void) { return SGPR_ABI_VERSION; }

extern "C" void sgpr_destroy(sgpr_handle h);
static void drop_graphs(sgpr_context* h);

static int upload(DevBuf& b, const void* src, size_t bytes) {
    SGPR_TRY(b.ensure(bytes ? bytes : 8));
    if (bytes) SGPR_CUDA(cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice));
    return SGPR_OK;
}

static bool is_pinned_host(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

static int upload_weights(sgpr_context* h, const double* mu_h, const double* mean_w_h, const double* choli_h,
                          const double* vscale_h, const int64_t* ind_first_h) {
    const int M = h->M, S = h->S;
    if (mu_h) {
        h->mu_host.assign(mu_h, mu_h + M);
        std::vector<double> mus(M);
        for (int p = 0; p < M; ++p) mus[p] = mu_h[h->ind_perm[p]];
        SGPR_TRY(upload(h->mu, mus.data(), sizeof(double) * M));
        std::vector<double> lone(SGPR_MAX_SPECIES, 0.0);
        for (int p = 0; p < M; ++p)
            if (h->ind_lone[p]) lone[h->ind_sp[p]] += h->lone_w * mus[p];
        SGPR_TRY(upload(h->lone_mu, lone.data(), sizeof(double) * SGPR_MAX_SPECIES));
    }
    if (mean_w_h) {
        h->mean_w.assign(mean_w_h, mean_w_h + S);
        h->mean_w.resize(SGPR_MAX_SPECIES, 0.0);
        SGPR_TRY(upload(h->mean_w_d, h->mean_w.data(), sizeof(double) * SGPR_MAX_SPECIES));
    }
    if (vscale_h) {
        h->vscale.assign(vscale_h, vscale_h + S);
        h->vscale.resize(SGPR_MAX_SPECIES, INFINITY);
        SGPR_TRY(upload(h->vscale_d, h->vscale.data(), sizeof(double) * SGPR_MAX_SPECIES));
    }
    if (choli_h) {
        // per central species: choli[:, columns of that species] (sorted inducing order), rows
        // zero-padded to ld_zt -> the B operand of the covloss GEMM (K contiguous)
        std::vector<double> c((size_t)S * M * h->ld_zt, 0.0);
        std::vector<double> clone(SGPR_MAX_SPECIES, 0.0);
        for (int s = 0; s < S; ++s) {
            const int m0 = h->m_first[s], m1 = h->m_first[s + 1];
            for (int k = 0; k < M; ++k) {
                double lone_sum = 0.0;
                for (int p = m0; p < m1; ++p) {
                    const double v = choli_h[(size_t)k * M + h->ind_perm[p]];
                    c[((size_t)s * M + k) * h->ld_zt + (p - m0)] = v;
                    if (h->ind_lone[p]) lone_sum += v;
                }
                // c / alpha of a neighbour-less atom: K row = lone_w x lone indicator, self kernel alpha = lone_w
                clone[s] += h->lone_w * lone_sum * lone_sum;
            }
        }
        SGPR_TRY(upload(h->choli_t, c.data(), sizeof(double) * c.size()));
        SGPR_TRY(upload(h->clone_d, clone.data(), sizeof(double) * SGPR_MAX_SPECIES));
        h->has_choli = true;
    }
    (void)ind_first_h;
    return SGPR_OK;
}

// Inducing set (a10): group the LCEs by central species, evaluate Z_hat with the atom kernels, build the per-species
// transposes.  Keeps host copies of the environments so that sgpr_append_inducing can extend the set.
static int set_inducing(sgpr_context* h, int M, const int32_t* ind_Z, const int64_t* ind_first, const double* ind_r,
                        const int32_t* ind_b) {
    // inducing set, grouped by central species
    DescParams& dp = h->dp;
    const int S = h->S;
    h->M = M;
    std::vector<int> sp_of(M);
    for (int m = 0; m < M; ++m) {
        const int z = ind_Z[m];
        if (z < 0 || z >= 128 || h->z_to_species[z] < 0) {
            set_error("inducing LCE %d: species Z=%d not in the species table", m, z);
            return SGPR_ERR_SPECIES;
        }
        sp_of[m] = h->z_to_species[z];
    }
    h->ind_perm.resize(M);
    for (int m = 0; m < M; ++m) h->ind_perm[m] = m;
    std::stable_sort(h->ind_perm.begin(), h->ind_perm.end(), [&](int a, int b) { return sp_of[a] < sp_of[b]; });
    for (int s = 0; s <= SGPR_MAX_SPECIES; ++s) h->m_first[s] = 0;
    for (int m = 0; m < M; ++m) h->m_first[sp_of[m] + 1]++;
    for (int s = 0; s < SGPR_MAX_SPECIES; ++s) h->m_first[s + 1] += h->m_first[s];
    int maxMs = 0;
    for (int s = 0; s < S; ++s) maxMs = std::max(maxMs, h->m_first[s + 1] - h->m_first[s]);
    h->ld_zt = std::max(16, (maxMs + 15) & ~15);
    h->ldg = h->ld_zt;
    h->ind_sp.resize(M);
    h->ind_lone.resize(M);
    std::vector<int> row_of(M);
    for (int p = 0; p < M; ++p) {
        const int m = h->ind_perm[p];
        row_of[m] = p;
        h->ind_sp[p] = sp_of[m];
        h->ind_lone[p] = (ind_first[m + 1] == ind_first[m]) ? 1 : 0;
    }
    SGPR_TRY(upload(h->ind_perm_d, h->ind_perm.data(), sizeof(int) * M));
    {
        std::vector<unsigned char> on(SGPR_MAX_SPECIES, 0);
        for (int s = 0; s < S; ++s) on[s] = (dp.central_enabled[s] && h->m_first[s + 1] > h->m_first[s]) ? 1 : 0;
        SGPR_TRY(upload(h->sp_on, on.data(), SGPR_MAX_SPECIES));
    }
    // environments -> device, evaluate Z_hat with the atom kernels
    SGPR_TRY(h->zhat.ensure(sizeof(double) * ((size_t)M + 1) * dp.ldp));
    SGPR_CUDA(cudaMemset(h->zhat.p, 0, sizeof(double) * ((size_t)M + 1) * dp.ldp));
    if (M > 0) {
        const int64_t nnz = ind_first[M];
        std::vector<unsigned char> esp((size_t)nnz + 1);
        for (int64_t k = 0; k < nnz; ++k) {
            const int z = ind_b[k];
            if (z < 0 || z >= 128 || h->z_to_species[z] < 0) {
                set_error("inducing neighbour species Z=%d not in the species table", z);
                    return SGPR_ERR_SPECIES;
            }
            esp[k] = (unsigned char)h->z_to_species[z];
        }
        std::vector<long long> first(M + 1);
        for (int m = 0; m <= M; ++m) first[m] = ind_first[m];
        DevBuf b_first, b_r, b_sp, b_row;
        SGPR_TRY(upload(b_first, first.data(), sizeof(long long) * (M + 1)));
        SGPR_TRY(upload(b_r, ind_r, sizeof(double) * 3 * nnz));
        SGPR_TRY(upload(b_sp, esp.data(), nnz));
        SGPR_TRY(upload(b_row, row_of.data(), sizeof(int) * M));
        int st = descriptor_forward_env(h, M, b_first.as<long long>(), b_r.as<double>(), b_sp.as<unsigned char>(),
                                        b_row.as<int>(), h->zhat.as<double>(), 0);
        if (st == SGPR_OK && cudaDeviceSynchronize() != cudaSuccess) {
            set_error("inducing descriptor kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
            st = SGPR_ERR_CUDA;
        }
        b_first.release();
        b_r.release();
        b_sp.release();
        b_row.release();
        if (st != SGPR_OK) return st;
    }
    // transposed copies per species for the back projection
    SGPR_TRY(h->zhat_t.ensure(sizeof(double) * (size_t)S * dp.D * h->ld_zt + 8));
    SGPR_CUDA(cudaMemset(h->zhat_t.p, 0, sizeof(double) * (size_t)S * dp.D * h->ld_zt + 8));
    for (int s = 0; s < S; ++s) {
        h->zt_off[s] = (size_t)s * dp.D * h->ld_zt;
        const int Ms = h->m_first[s + 1] - h->m_first[s];
        if (Ms == 0) continue;
        dim3 grid((dp.D + 31) / 32, (h->ld_zt + 31) / 32), block(32, 8);
        transpose_zhat_kernel<<<grid, block>>>(dp.D, dp.ldp, h->m_first[s], Ms, h->ld_zt, h->zhat.as<double>(),
                                               h->zhat_t.as<double>() + h->zt_off[s]);
    }
    SGPR_CUDA(cudaDeviceSynchronize());
    {   // caller's order copies for the lone-lone kernel term
        std::vector<int> sp_orig(M + 1);
        std::vector<unsigned char> lone_orig(M + 1);
        for (int p = 0; p < M; ++p) {
            sp_orig[h->ind_perm[p]] = h->ind_sp[p];
            lone_orig[h->ind_perm[p]] = h->ind_lone[p];
        }
        SGPR_TRY(upload(h->ind_sp_d, sp_orig.data(), sizeof(int) * M));
        SGPR_TRY(upload(h->ind_lone_d, lone_orig.data(), M));
    }
    {   // host copies (no-op when called with the copies themselves)
        const int64_t nnz = M > 0 ? ind_first[M] : 0;
        std::vector<int32_t> zc(ind_Z, ind_Z + M), bc(ind_b, ind_b + nnz);
        std::vector<int64_t> fc(ind_first, ind_first + (M > 0 ? M + 1 : 0));
        std::vector<double> rc(ind_r, ind_r + 3 * nnz);
        if (M == 0) fc.assign(1, 0);
        h->ind_Z_host.swap(zc);
        h->ind_b_host.swap(bc);
        h->ind_first_host.swap(fc);
        h->ind_r_host.swap(rc);
    }
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_create(const sgpr_model_desc* d, sgpr_handle* out) {
    if (!d || !out) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device available: libsgpr_b200 has no CPU fallback");
        return SGPR_ERR_NO_DEVICE;
    }
    if (d->device < 0 || d->device >= ndev) {
        set_error("device %d out of range (have %d)", d->device, ndev);
        return SGPR_ERR_INVALID;
    }
    if (d->lmax < 0 || d->lmax > kMaxL || d->nmax < 0 || d->nmax + 1 > kMaxNB) {
        set_error("unsupported lmax=%d (max %d) / nmax=%d (max %d)", d->lmax, kMaxL, d->nmax, kMaxNB - 1);
        return SGPR_ERR_INVALID;
    }
    if (d->n_species < 1 || d->n_species > SGPR_MAX_SPECIES) {
        set_error("n_species=%d not in 1..%d", d->n_species, SGPR_MAX_SPECIES);
        return SGPR_ERR_INVALID;
    }
    if (!(d->rc > 0) || !(d->xi > 0) || d->M < 0) {
        set_error("invalid rc/xi/M");
        return SGPR_ERR_INVALID;
    }
    if (d->M > 0 && (!d->mu_h || !d->ind_Z_h || !d->ind_first_h)) {
        set_error("M = %d inducing LCEs but mu_h / ind_Z_h / ind_first_h is null", d->M);
        return SGPR_ERR_INVALID;
    }
    SGPR_CUDA(cudaSetDevice(d->device));
    sgpr_context* h = new sgpr_context();
    // any error return below destroys the half-built context (stream, events, device buffers)
    struct Guard {
        sgpr_context* h;
        ~Guard() {
            if (h) sgpr_destroy(h);
        }
    } guard{h};
    h->device = d->device;
    cudaDeviceProp prop;
    SGPR_CUDA(cudaGetDeviceProperties(&prop, d->device));
    h->sm_count = prop.multiProcessorCount;
    SGPR_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 6; ++i) SGPR_CUDA(cudaEventCreate(&h->ev[i]));
    SGPR_TRY(upload_harm_coef());

    DescParams& dp = h->dp;
    const int S = d->n_species;
    h->S = S;
    dp.lmax = d->lmax;
    dp.nb = d->nmax + 1;
    dp.L2 = (d->lmax + 1) * (d->lmax + 1);
    dp.S = S;
    dp.A = S * dp.nb;
    dp.L2p = dp.L2 | 1;
    dp.ncomp = dp.nb * dp.L2;
    dp.csize = dp.A * dp.L2p;
    const int L = d->lmax + 1;
    dp.D = dp.A * (dp.A + 1) / 2 * L;
    dp.ldp = (dp.D + 15) & ~15;
    dp.normalize = d->normalize ? 1 : 0;
    dp.rc = d->rc;
    dp.rc_inv = 1.0 / d->rc;
    if (dp.A > 255) {
        set_error("S*(nmax+1) = %d exceeds 255", dp.A);
        return SGPR_ERR_INVALID;
    }
    SGPR_TRY(descriptor_check_size(dp));
    for (int i = 0; i < 128; ++i) h->z_to_species[i] = -1;
    for (int s = 0; s < SGPR_MAX_SPECIES; ++s) {
        dp.radii[s] = 1.0;
        dp.rinv[s] = 1.0;
        dp.central_enabled[s] = 0;
        dp.nbr_enabled[s] = 0;
        h->species_Z[s] = -1;
    }
    for (int s = 0; s < S; ++s) {
        const int z = d->species_Z[s];
        if (z < 0 || z >= 128 || h->z_to_species[z] >= 0 || !(d->radii[s] > 0)) {
            set_error("bad species table entry %d (Z=%d, radius=%g)", s, z, d->radii[s]);
                return SGPR_ERR_INVALID;
        }
        h->species_Z[s] = z;
        h->z_to_species[z] = s;
        dp.radii[s] = d->radii[s];
        dp.rinv[s] = 1.0 / d->radii[s];
        dp.central_enabled[s] = d->central_enabled[s] ? 1 : 0;
        dp.nbr_enabled[s] = d->neighbor_enabled[s] ? 1 : 0;
    }
    h->xi = d->xi;
    h->lone_w = d->lone_weight > 0 ? d->lone_weight : (d->lone_weight < 0 ? 0.0 : 1.0);
    h->xi_int = (d->xi == std::floor(d->xi) && d->xi >= 1 && d->xi <= 64) ? (int)d->xi : -1;
    SGPR_TRY(upload(h->ztab, h->z_to_species, sizeof(int) * 128));
    SGPR_TRY(h->errflag.ensure(sizeof(int) * 4));
    SGPR_TRY(h->status_d.ensure(sizeof(long long) * 8));
    SGPR_CUDA(cudaMemset(h->status_d.p, 0, sizeof(long long) * 8));
    SGPR_CUDA(cudaMallocHost((void**)&h->status_pinned, sizeof(long long) * 8));
    memset(h->status_pinned, 0, sizeof(long long) * 8);
    SGPR_TRY(h->row_first_d.ensure(sizeof(int) * (SGPR_MAX_SPECIES + 2)));
    SGPR_CUDA(cudaMemset(h->row_first_d.p, 0, sizeof(int) * (SGPR_MAX_SPECIES + 2)));

    // packed-entry tables
    {
        std::vector<unsigned> ptab(dp.D);
        std::vector<double> nnlk(dp.D);
        for (int a = 0; a < dp.A; ++a)
            for (int b = a; b < dp.A; ++b) {
                const int tri = a * dp.A - (a * (a - 1)) / 2 + (b - a);
                const int na = a % dp.nb, nbb = b % dp.nb;
                for (int l = 0; l < L; ++l) {
                    ptab[tri * L + l] = (unsigned)a | ((unsigned)b << 8) | ((unsigned)l << 16);
                    nnlk[tri * L + l] = std::sqrt(anl(na, l) * anl(nbb, l)) * (a == b ? 1.0 : std::sqrt(2.0));
                }
            }
        SGPR_TRY(upload(h->ptab, ptab.data(), sizeof(unsigned) * dp.D));
        SGPR_TRY(upload(h->nnlk, nnlk.data(), sizeof(double) * dp.D));
        // chain-rule table of the back projection: dp/dc picks up kappa*nnl and a factor 2 on a == b
        std::vector<double> ttab(dp.ldp, 0.0);
        for (int e = 0; e < dp.D; ++e) ttab[e] = nnlk[e] * (((ptab[e] & 0xff) == ((ptab[e] >> 8) & 0xff)) ? 2.0 : 1.0);
        SGPR_TRY(upload(h->ttab, ttab.data(), sizeof(double) * dp.ldp));
    }

    {
        const int st_ind = set_inducing(h, d->M, d->ind_Z_h, d->ind_first_h, d->ind_r_h, d->ind_b_h);
        if (st_ind != SGPR_OK) {
                return st_ind;
        }
    }
    std::vector<double> zeros(SGPR_MAX_SPECIES, 0.0), infs(SGPR_MAX_SPECIES, INFINITY);
    int st = upload_weights(h, d->mu_h, d->mean_w_h ? d->mean_w_h : zeros.data(), d->choli_h,
                            d->vscale_h ? d->vscale_h : infs.data(), nullptr);
    if (st != SGPR_OK) {
        return st;
    }
    {   // GEMM engine: tcgen05 int8-sliced (default, needs normalised descriptors) or FP64 DMMA
        const char* nlm = getenv("SGPR_NL");
        h->nl_mode = !nlm ? 0 : strcmp(nlm, "warp") == 0 ? 1 : strcmp(nlm, "bins") == 0 ? 2 : 0;
        const char* lean = getenv("SGPR_NL_LEAN");
        h->nl_lean = !(lean && atoi(lean) == 0);
        const char* gr = getenv("SGPR_GRAPH");
        h->use_graph = !(gr && atoi(gr) == 0);
        const char* eng = getenv("SGPR_GEMM");
        const char* trs = getenv("SGPR_I8_TR");
        h->use_i8 = dp.normalize && !(eng && strcmp(eng, "dmma") == 0);
        h->i8_tr = (trs && atoi(trs) == 8) ? 8 : 7;
        const char* tr2 = getenv("SGPR_I8_TR2");   // back projection (forces only): like the kernel matrix, or 6 / 7 / 8
        h->i8_tr2 = tr2 ? (atoi(tr2) == 8 ? 8 : atoi(tr2) == 6 ? 6 : 7) : h->i8_tr;
        const char* c2 = getenv("SGPR_I8_CTA2");
        h->i8_cta2 = c2 && atoi(c2) == 1;
        const char* epw = getenv("SGPR_I8_EPW");
        h->i8_epw = epw ? atoi(epw) : 0;
        const char* nss = getenv("SGPR_I8_NS");
        h->i8_ns = (nss && atoi(nss) == 5) ? 5 : 6;
        if (h->use_i8) {
            st = i8_prepare_model(h, false);
            if (st == SGPR_OK) st = i8_prepare_covloss(h);
            if (st != SGPR_OK) {
                        return st;
            }
        }
    }
    memset(&h->stats, 0, sizeof(h->stats));
    h->stats.d_packed = dp.D;
    h->stats.d_full = dp.A * dp.A * L;
    guard.h = nullptr;
    *out = h;
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) void sgpr_destroy(sgpr_handle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    drop_graphs(h);
    DevBuf* bufs[] = {&h->zhat, &h->zhat_t, &h->mu, &h->lone_mu, &h->ptab, &h->nnlk, &h->ztab, &h->errflag,
                      &h->ind_perm_d, &h->sp_on, &h->ind_sp_d, &h->ind_lone_d, &h->mean_w_d, &h->cnt, &h->cstart,
                      &h->rstart, &h->keyrank, &h->atoms, &h->order, &h->rowof, &h->active_list, &h->nl_cnt,
                      &h->nl_first, &h->nl_pairs, &h->scan_tmp, &h->phat, &h->cbuf, &h->pnorm, &h->sflag, &h->gmat,
                      &h->gvec, &h->epart, &h->wpart, &h->fcell, &h->misc, &h->stage_pos, &h->stage_z, &h->stage_out,
                      &h->rowmap, &h->owned, &h->shard_tmp, &h->row_owned, &h->choli_t, &h->vscale_d, &h->clone_d,
                      &h->kcmat, &h->cpart, &h->nl_masks, &h->erow_part, &h->erow, &h->prow, &h->ttab, &h->z8, &h->zt8, &h->p8, &h->g8, &h->i8_probs, &h->k8, &h->c8, &h->crs, &h->nl_run, &h->cov_nk, &h->row_first_d, &h->status_d, &h->p2p_local, &h->i8_probs2,
                      &h->b_geom, &h->b_first, &h->b_bins, &h->b_cell, &h->b_err, &h->astr, &h->wenv, &h->jsel, &h->kscr,
                      &h->md_pos, &h->md_mom, &h->md_F, &h->md_beta, &h->md_ew, &h->md_part,
                      &h->rx_pos, &h->rx_vel, &h->rx_F, &h->rx_beta, &h->rx_ew, &h->rx_part};
    for (DevBuf* b : bufs) b->release();
    if (h->pinned) cudaFreeHost(h->pinned);
    if (h->i8_probs_pinned) cudaFreeHost(h->i8_probs_pinned);
    if (h->status_pinned) cudaFreeHost(h->status_pinned);
    if (h->i8_probs2_pinned) cudaFreeHost(h->i8_probs2_pinned);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    for (int i = 0; i < 6; ++i)
        if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    delete h;
}

extern "C" __attribute__((visibility("default"))) int sgpr_set_weights(sgpr_handle h, const double* mu_h, const double* mean_w_h, const double* choli_h,
                                const double* vscale_h) {
    if (!h) {
        set_error("null handle");
        return SGPR_ERR_INVALID;
    }
    SGPR_CUDA(cudaSetDevice(h->device));
    SGPR_CUDA(cudaDeviceSynchronize());
    drop_graphs(h);   // weight buffers may be reallocated
    h->warm_ok = false;
    SGPR_TRY(upload_weights(h, mu_h, mean_w_h, choli_h, vscale_h, nullptr));
    if (mu_h && h->use_i8) SGPR_TRY(i8_prepare_model(h, true));
    if (choli_h && h->use_i8) SGPR_TRY(i8_prepare_covloss(h));
    return SGPR_OK;
}

// Extend the inducing set (regression/gppotential.py:888-940 add_inducing / calculator/active.py:842-929
// update_inducing): new LCEs are appended after the existing ones (caller's order), all model-side operands are
// rebuilt, and the weights -- whose sizes change with M -- are replaced in the same call.
extern "C" __attribute__((visibility("default"))) int sgpr_append_inducing(sgpr_handle h, int32_t n_new, const int32_t* ind_Z_h,
                                    const int64_t* ind_first_h, const double* ind_r_h, const int32_t* ind_b_h,
                                    const double* mu_h, const double* choli_h) {
    if (!h || n_new < 0 || !mu_h || (n_new > 0 && (!ind_Z_h || !ind_first_h))) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    SGPR_CUDA(cudaSetDevice(h->device));
    SGPR_CUDA(cudaDeviceSynchronize());
    const int M0 = h->M, M1 = M0 + n_new;
    const int64_t nnz0 = h->ind_first_host.empty() ? 0 : h->ind_first_host[M0];
    const int64_t nnz_new = n_new > 0 ? ind_first_h[n_new] - ind_first_h[0] : 0;
    if (nnz_new < 0 || (nnz_new > 0 && (!ind_r_h || !ind_b_h))) {
        set_error("bad CSR of the new inducing environments");
        return SGPR_ERR_INVALID;
    }
    std::vector<int32_t> Z(h->ind_Z_host), b(h->ind_b_host);
    std::vector<int64_t> first(h->ind_first_host);
    std::vector<double> r(h->ind_r_host);
    if (first.empty()) first.assign(1, 0);
    const std::vector<int32_t> Z0(Z), b0(b);
    const std::vector<int64_t> first0(first);
    const std::vector<double> r0(r);
    for (int m = 0; m < n_new; ++m) {
        Z.push_back(ind_Z_h[m]);
        first.push_back(nnz0 + (ind_first_h[m + 1] - ind_first_h[0]));
    }
    const int64_t o = n_new > 0 ? ind_first_h[0] : 0;
    b.insert(b.end(), ind_b_h + o, ind_b_h + o + nnz_new);
    r.insert(r.end(), ind_r_h + 3 * o, ind_r_h + 3 * (o + nnz_new));
    int st = set_inducing(h, M1, Z.data(), first.data(), r.data(), b.data());
    if (st != SGPR_OK) {   // e.g. an unknown species: keep the old model usable
        const std::string msg = sgpr_last_error();
        set_inducing(h, M0, Z0.data(), first0.data(), r0.data(), b0.data());
        set_error("%s", msg.c_str());
        return st;
    }
    h->has_choli = false;
    h->fwd_valid = false;
    h->warm_ok = false;
    drop_graphs(h);
    h->i8_cap_rows = 0;   // the K padding of the per-step digit buffers follows max M_s
    SGPR_TRY(upload_weights(h, mu_h, nullptr, choli_h, nullptr, nullptr));
    if (h->use_i8) {
        SGPR_TRY(i8_prepare_model(h, false));
        SGPR_TRY(i8_prepare_covloss(h));
    }
    return SGPR_OK;
}

// =====================================================================================
// pipeline
// =====================================================================================
static int stage_front(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                       const int32_t* pbc_h, cudaStream_t st, Geom* g, int rank = 0, int world = 1, bool i8 = false,
                       bool with_halo = true, bool with_k8 = false, bool warm = false) {
    h->use_i8_now = i8 && h->use_i8;
    if (!warm) h->stats.i8_ops = 0.0;      // warm steps: the work counters of the sizing step stay (same shape)
    h->fwd_valid = false;
    // geometry -> cell sort -> neighbour list -> descriptors (rows in species-major order)
    if (N < 0 || N > 0x7fffff00ll) {
        set_error("bad atom count");
        return SGPR_ERR_INVALID;
    }
    h->stats.n_atoms = N;
    h->stats.kernel_launches = 0;
    if (!warm) h->stats.gemm_flops = 0.0;
    h->last_N = N;
    SGPR_TRY(build_geometry(h, N, pos_d, cell_h, pbc_h, st, g));
    h->last_geom = *g;
    if (h->timing) cudaEventRecord(h->ev[0], st);
    nvtxRangePushA("sgpr:nl");
    struct PopOnExit {
        bool armed = true;
        ~PopOnExit() {
            if (armed) nvtxRangePop();
        }
    } nl_range;
    SGPR_TRY(cell_sort(h, N, pos_d, Z_d, *g, st));
    // neighbour list (+ halo when sharded); species row ranges come back with the pair count
    int64_t n_pairs = 0;
    if (world == 1)
        SGPR_TRY(neighbor_build(h, N, *g, st, &n_pairs, warm));  // sizing step: synchronises the stream
    else
        SGPR_TRY(neighbor_build_sharded(h, N, *g, rank, world, st, &n_pairs, with_halo, warm));
    h->stats.n_active = h->n_active;
    if (!warm) h->stats.n_pairs = n_pairs;
    nl_range.armed = false;
    nvtxRangePop();
    NvtxRange desc_range("sgpr:desc");
    if (h->timing) cudaEventRecord(h->ev[1], st);
    SGPR_TRY(h->phat.ensure(sizeof(double) * ((size_t)h->n_active + 1) * h->dp.ldp));
    if (h->use_i8_now) SGPR_TRY(i8_ensure_step_buffers(h, (size_t)h->n_active, with_k8));
    SGPR_TRY(descriptor_forward_atoms(h, *g, st));
    if (h->timing) cudaEventRecord(h->ev[2], st);
    return SGPR_OK;
}

static bool warm_possible(sgpr_handle h, int64_t N, const int32_t* pbc_h, int32_t rank, int32_t world, bool p2p, bool beta) {
    const bool halo_mode = world > 1 && !p2p;
    return h->use_i8 && pbc_h[0] && pbc_h[1] && pbc_h[2] && !halo_mode && h->warm_ok && N == h->warm_N &&
           rank == h->warm_rank && world == h->warm_world && beta == h->warm_beta;
}

constexpr int kRowEnergyGrid = 128;   // blocks (= energy partials) of row_energy_kernel

// energy partials per row of each central species (0 where the species has no usable inducing points)
static RowSpecies row_species(sgpr_context* h, int* max_part) {
    RowSpecies rs{};
    rs.S = h->S;
    for (int s = 0; s < h->S; ++s) {
        const int Ms = h->m_first[s + 1] - h->m_first[s];
        rs.n_part[s] = (Ms > 0 && h->dp.central_enabled[s]) ? (h->use_i8_now ? i8_energy_parts(Ms) : gemm_energy_parts(Ms)) : 0;
        if (rs.n_part[s] > *max_part) *max_part = rs.n_part[s];
    }
    return rs;
}

// kernel matrix of the step's rows -> local energies erow (+ block partials epart) -> back projection gvec = dE/dq_hat
static int gemm_stage(sgpr_context* h, cudaStream_t st, const RowSpecies& rs, bool with_beta) {
    const size_t nrows = (size_t)h->n_active + 1;
    nvtxRangePushA("sgpr:gemm");
    struct PopGemm {
        bool armed = true;
        ~PopGemm() {
            if (armed) nvtxRangePop();
        }
    } gemm_range;
    if (h->use_i8_now)
        SGPR_TRY(i8_kernel_matrix(h, st, with_beta));
    else
        SGPR_TRY(gemm_kernel_matrix(h, nullptr, 0, nullptr, with_beta, st));
    row_energy_kernel<<<kRowEnergyGrid, 256, 0, st>>>((int)h->n_active, rs, h->row_first_d.as<int>(), h->erow_part.as<double>(),
                                                      (int)nrows, h->active_all ? nullptr : h->row_owned.as<unsigned char>(),
                                                      h->erow.as<double>(), h->epart.as<double>());
    h->stats.kernel_launches += 1;
    if (h->use_i8_now)
        SGPR_TRY(i8_back_projection(h, st));
    else
        SGPR_TRY(gemm_back_projection(h, st));
    if (h->timing) cudaEventRecord(h->ev[3], st);
    gemm_range.armed = false;
    nvtxRangePop();
    return SGPR_OK;
}

// covloss of the step's environments into beta_d [N] (caller's order)
static int covloss_stage(sgpr_context* h, cudaStream_t st, int64_t N, const int* active, const unsigned char* owned,
                         double* beta_d) {
    const size_t nrows = (size_t)h->n_active + 1;
    NvtxRange covloss_range("sgpr:covloss");
    const int n_part = h->use_i8_now ? i8_covloss_parts(h) : gemm_covloss_parts(h);
    SGPR_TRY(h->cpart.ensure(sizeof(double) * (size_t)n_part * nrows));
    SGPR_CUDA(cudaMemsetAsync(beta_d, 0, sizeof(double) * (size_t)N, st));
    if (h->use_i8_now)
        SGPR_TRY(i8_covloss(h, (int64_t)nrows, st));
    else
        SGPR_TRY(gemm_covloss(h, (int64_t)nrows, st));
    if (h->n_active > 0) {
        SGPR_TRY(h->misc.ensure(sizeof(int) * SGPR_MAX_SPECIES));
        SGPR_CUDA(cudaMemcpyAsync(h->misc.p, h->dp.central_enabled, sizeof(int) * SGPR_MAX_SPECIES,
                                  cudaMemcpyHostToDevice, st));
        beta_finish_kernel<<<h->sm_count * 2, 256, 0, st>>>(
            (int)h->n_active, active, h->atoms.as<AtomRec>(), h->rowof.as<int>() + (N + 1), h->nl_first.as<long long>(),
            owned, h->sp_on.as<unsigned char>(), h->misc.as<int>(), h->cpart.as<double>(), n_part, (int)nrows,
            h->clone_d.as<double>(), h->vscale_d.as<double>(), h->prow.as<double>(), h->dp.normalize, h->xi, beta_d);
        h->stats.kernel_launches += 1;
    }
    SGPR_CUDA(cudaGetLastError());
    return SGPR_OK;
}

// stage times of a call from the events ev[0..4] recorded on its way and ev[5] recorded here (synchronises)
static int read_stage_times(sgpr_context* h, cudaStream_t st) {
    cudaEventRecord(h->ev[5], st);
    SGPR_CUDA(cudaEventSynchronize(h->ev[5]));
    cudaEventElapsedTime(&h->stats.ms_nl, h->ev[0], h->ev[1]);
    cudaEventElapsedTime(&h->stats.ms_desc, h->ev[1], h->ev[2]);
    cudaEventElapsedTime(&h->stats.ms_gemm, h->ev[2], h->ev[3]);
    cudaEventElapsedTime(&h->stats.ms_force, h->ev[3], h->ev[4]);
    cudaEventElapsedTime(&h->stats.ms_beta, h->ev[4], h->ev[5]);
    cudaEventElapsedTime(&h->stats.ms_total, h->ev[0], h->ev[5]);
    return SGPR_OK;
}

static int predict_body(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                        const int32_t* pbc_h, int32_t rank, int32_t world, void* stream, double* E_d, double* F_d,
                        double* W_d, double* beta_d, uint8_t* owned_d, const uint64_t* peer_f_h, bool allow_warm,
                        const P2PStep* px = nullptr) {
    if (!h || !cell_h || !pbc_h || !E_d || (!F_d && !peer_f_h) || !W_d || (N > 0 && (!pos_d || !Z_d))) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    if (peer_f_h && world > SGPR_MAX_RANKS) {
        set_error("peer-memory force exchange supports at most %d ranks", SGPR_MAX_RANKS);
        return SGPR_ERR_INVALID;
    }
    if (world < 1 || rank < 0 || rank >= world) {
        set_error("bad rank/world (%d/%d)", rank, world);
        return SGPR_ERR_INVALID;
    }
    if (beta_d && !h->has_choli) {
        set_error("covloss requested but the model has no choli");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    Geom g;
    double* E_out = E_d;
    double* W_out = W_d;
    if (px) {
        // fused exchange step: the accumulation buffer of the NEXT step is cleared now (its last readers finished in
        // the previous step of this stream; remote ranks touch it only after they have seen this step's flag)
        SGPR_TRY(h->p2p_local.ensure(sizeof(double) * 16 + sizeof(long long) * 2));
        if (!h->p2p_counter_init) {   // (always a sizing step: never inside a graph capture)
            SGPR_CUDA(cudaStreamSynchronize(st));
            SGPR_CUDA(cudaMemset(h->p2p_local.p, 0, sizeof(double) * 16 + sizeof(long long) * 2));
            h->p2p_counter_init = true;
        }
        p2p_zero_next_kernel<<<h->sm_count, 256, 0, st>>>(px->own_base, px->stride, 3 * ((long long)N + 1),
                                                          reinterpret_cast<const long long*>(h->p2p_local.as<double>() + 16));
        E_d = h->p2p_local.as<double>();        // this rank's partial sums
        W_d = h->p2p_local.as<double>() + 1;
    }
    // Sync-free ("warm") step: every size the host needs was fixed by an earlier sizing step of the same shape; the
    // pair count, the species row ranges and the error flags stay on the device (nl.cu: nl_status_kernel).
    const bool halo_mode = world > 1 && peer_f_h == nullptr;
    const bool shape_ok = h->use_i8 && pbc_h[0] && pbc_h[1] && pbc_h[2] && !halo_mode;
    const bool warm = allow_warm && warm_possible(h, N, pbc_h, rank, world, peer_f_h != nullptr, beta_d != nullptr);
    h->step_was_warm = warm;
    SGPR_TRY(stage_front(h, N, pos_d, Z_d, cell_h, pbc_h, st, &g, rank, world, /*i8=*/true,
                         /*with_halo=*/peer_f_h == nullptr, /*with_k8=*/beta_d != nullptr, warm));
    if (h->use_i8_now) SGPR_TRY(i8_setup_step(h, st));
    PeerForces peers{};
    if (peer_f_h) {
        peers.world = world;
        for (int r = 0; r < world; ++r) {
            peers.peer_f[r] = (double*)(uintptr_t)peer_f_h[r];
            peers.bounds[r] = (int)((N * r) / world);
        }
        peers.bounds[world] = (int)N;
        peers.parity_src = px ? reinterpret_cast<const long long*>(h->p2p_local.as<double>() + 16) : nullptr;
        peers.parity_stride = px ? px->stride : 0;
        h->p2p_rank = rank;
    }
    const unsigned char* owned = h->active_all ? nullptr : h->owned.as<unsigned char>();
    const int* active = h->active_all ? nullptr : h->active_list.as<int>();
    const int grid_g = kRowEnergyGrid;
    const int nblk_b = backward_grid(h);
    const int nblk_x = 64;
    const size_t nrows = (size_t)h->n_active + 1;
    int max_part = 1;
    const RowSpecies rs = row_species(h, &max_part);
    SGPR_TRY(h->erow_part.ensure(sizeof(double) * (size_t)max_part * nrows));
    SGPR_TRY(h->erow.ensure(sizeof(double) * nrows));
    if (!h->use_i8_now) SGPR_TRY(h->gmat.ensure(sizeof(double) * nrows * h->ldg));
    SGPR_TRY(h->gvec.ensure(sizeof(double) * nrows * h->dp.ldp));
    SGPR_TRY(h->epart.ensure(sizeof(double) * ((size_t)grid_g + nblk_x)));
    SGPR_TRY(h->wpart.ensure(sizeof(double) * 9 * nblk_b));
    SGPR_TRY(h->fcell.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    // every partial is written by its producer (row_energy_kernel, atom_terms_kernel, the backward kernel: one entry per
    // block, grids fixed) unless a rank has nothing to do
    if (N == 0 || h->n_active == 0) {
        SGPR_CUDA(cudaMemsetAsync(h->epart.p, 0, sizeof(double) * ((size_t)grid_g + nblk_x), st));
        SGPR_CUDA(cudaMemsetAsync(h->wpart.p, 0, sizeof(double) * 9 * nblk_b, st));
    }
    if (!peer_f_h) SGPR_CUDA(cudaMemsetAsync(h->fcell.p, 0, sizeof(double) * 3 * ((size_t)N + 1), st));
    if (beta_d && !h->use_i8_now) SGPR_TRY(h->kcmat.ensure(sizeof(double) * nrows * h->ldg));
    SGPR_TRY(gemm_stage(h, st, rs, beta_d != nullptr));
    NvtxRange force_range("sgpr:force");
    SGPR_TRY(descriptor_backward_atoms(h, g, owned, st, peer_f_h ? &peers : nullptr));
    if (peer_f_h && N > 0) {
        p2p_push_kernel<<<h->sm_count * 2, 256, 0, st>>>(3 * (long long)N, peers, h->p2p_rank);
        h->stats.kernel_launches += 1;
    }
    if (N > 0) {
        atom_terms_kernel<<<nblk_x, 256, 0, st>>>(N, (int)h->n_active, active, h->atoms.as<AtomRec>(),
                                                  h->nl_first.as<long long>(), owned, h->mean_w_d.as<double>(),
                                                  h->lone_mu.as<double>(),
                                                  h->epart.as<double>() + (size_t)grid_g);
        if (!peer_f_h)
            scatter_forces_kernel<<<(int)((N + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(), h->fcell.as<double>(),
                                                                          owned, F_d, owned_d);
    }
    final_reduce_kernel<<<1, 320, 0, st>>>(grid_g, h->epart.as<double>(), nblk_x,
                                           h->epart.as<double>() + (size_t)grid_g, nblk_b,
                                           h->wpart.as<double>(), E_d, W_d);
    h->stats.kernel_launches += 3;
    SGPR_CUDA(cudaGetLastError());
    if (h->timing) cudaEventRecord(h->ev[4], st);
    if (!warm) h->stats.covloss_flops = 0.0;
    if (beta_d) SGPR_TRY(covloss_stage(h, st, N, active, owned, beta_d));
    if (px) {
        long long* counter = reinterpret_cast<long long*>(h->p2p_local.as<double>() + 16);
        p2p_publish_wait_kernel<<<1, 32, 0, st>>>(rank, world, px->peers, h->p2p_local.as<double>(), counter, E_out, W_out,
                                                  h->status_d.as<long long>());
        if (N > 0)
            scatter_forces_kernel<<<(int)((N + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(), px->own_base,
                                                                          h->owned.as<unsigned char>(), px->F_d, px->owned_d,
                                                                          counter, px->stride);
        h->stats.kernel_launches += 2;
        SGPR_CUDA(cudaGetLastError());
    }
    if (warm) {
        // the step's status (pair count, validity) follows the results to the host; nobody waits for it here
        SGPR_CUDA(cudaMemcpyAsync(h->status_pinned, h->status_d.p, sizeof(long long) * 8, cudaMemcpyDeviceToHost, st));
    } else if (shape_ok) {
        h->warm_ok = true;
        h->warm_N = N;
        h->warm_rank = rank;
        h->warm_world = world;
        h->warm_beta = beta_d != nullptr;
    } else {
        h->warm_ok = false;
    }
    if (h->timing) SGPR_TRY(read_stage_times(h, st));
    return SGPR_OK;
}

// A warm step is the same launch sequence with the same arguments every time (same shape, same buffers, same cell):
// it is captured ONCE into a CUDA graph and replayed with a single cudaGraphLaunch afterwards -- ~30 kernel launches,
// memsets and the status copy collapse into one submission, which is what bounds small systems and multi-GPU shards.
// Graphs are keyed by everything that is baked into the nodes.
static int predict_impl(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                        const int32_t* pbc_h, int32_t rank, int32_t world, void* stream, double* E_d, double* F_d,
                        double* W_d, double* beta_d, uint8_t* owned_d, const uint64_t* peer_f_h, bool allow_warm,
                        const P2PStep* px = nullptr) {
    if (!h || !pbc_h || !cell_h || !h->use_graph || h->timing || !allow_warm || world > SGPR_MAX_RANKS ||
        !warm_possible(h, N, pbc_h, rank, world, peer_f_h != nullptr, beta_d != nullptr))
        return predict_body(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, F_d, W_d, beta_d, owned_d, peer_f_h, allow_warm, px);
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    sgpr_context::GraphKey key{};
    key.N = N;
    key.rank = rank;
    key.world = world;
    key.stream = stream;
    key.ptr[0] = pos_d; key.ptr[1] = Z_d; key.ptr[2] = E_d; key.ptr[3] = F_d; key.ptr[4] = W_d; key.ptr[5] = beta_d; key.ptr[6] = owned_d;
    for (int r = 0; r < SGPR_MAX_RANKS; ++r) key.peer[r] = (peer_f_h && r < world) ? peer_f_h[r] : 0;
    for (int i = 0; i < 9; ++i) key.cell[i] = cell_h[i];
    if (px) {
        key.px_on = 1;
        key.px_ptr[0] = px->F_d;
        key.px_ptr[1] = px->owned_d;
        key.px_ptr[2] = px->own_base;
        for (int r = 0; r < SGPR_MAX_RANKS; ++r) key.px_mail[r] = (uint64_t)(uintptr_t)px->peers.mail[r];
    }
    // a workspace was reallocated since the graphs were captured (e.g. a larger structure or a batch in between):
    // their nodes point at freed memory
    const unsigned long long gen = buf_generation();
    if (gen != h->graph_gen) {
        drop_graphs(h);
        h->graph_gen = gen;
    }
    for (auto& e : h->graphs) {
        if (memcmp(&e.key, &key, sizeof(key)) == 0) {
            e.stamp = ++h->graph_clock;
            h->step_was_warm = true;
            h->stats.kernel_launches = e.launches;
            SGPR_CUDA(cudaGraphLaunch(e.exec, st));
            return SGPR_OK;
        }
    }
    // first warm step of this key: record it
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
        cudaGetLastError();   // e.g. the legacy default stream cannot be captured: run the step directly
        return predict_body(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, F_d, W_d, beta_d, owned_d, peer_f_h, allow_warm, px);
    }
    const int rc = predict_body(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, F_d, W_d, beta_d, owned_d, peer_f_h, allow_warm, px);
    const cudaError_t ce = cudaStreamEndCapture(st, &graph);
    if (rc != SGPR_OK || ce != cudaSuccess || !graph || !h->step_was_warm) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        h->use_graph = false;   // something in the sequence is not capturable here: plain launches from now on
        h->warm_ok = false;     // (whatever was enqueued during the failed capture never ran)
        if (rc != SGPR_OK) return rc;
        return predict_body(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, F_d, W_d, beta_d, owned_d, peer_f_h, false, px);
    }
    cudaGraphExec_t exec = nullptr;
    if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
        cudaGraphDestroy(graph);
        cudaGetLastError();
        h->use_graph = false;
        h->warm_ok = false;
        return predict_body(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, F_d, W_d, beta_d, owned_d, peer_f_h, false, px);
    }
    cudaGraphDestroy(graph);
    if (h->graphs.size() >= 16) {   // evict the least recently used entry
        size_t lru = 0;
        for (size_t i = 1; i < h->graphs.size(); ++i)
            if (h->graphs[i].stamp < h->graphs[lru].stamp) lru = i;
        cudaGraphExecDestroy(h->graphs[lru].exec);
        h->graphs.erase(h->graphs.begin() + lru);
    }
    sgpr_context::GraphEntry e;
    e.key = key;
    e.exec = exec;
    e.stamp = ++h->graph_clock;
    e.launches = h->stats.kernel_launches;
    h->graphs.push_back(e);
    SGPR_CUDA(cudaGraphLaunch(exec, st));
    return SGPR_OK;
}

static void drop_graphs(sgpr_context* h) {
    for (auto& e : h->graphs) cudaGraphExecDestroy(e.exec);
    h->graphs.clear();
    drop_driver_graphs(h);
}

bool sgpr::md_warm_possible(sgpr_context* h, int64_t N, const int32_t* pbc_h, bool beta) {
    return warm_possible(h, N, pbc_h, 0, 1, false, beta);
}

int sgpr::md_predict(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                     const int32_t* pbc_h, cudaStream_t st, double* E_d, double* F_d, double* W_d, double* beta_d, bool graph) {
    if (graph) return predict_impl(h, N, pos_d, Z_d, cell_h, pbc_h, 0, 1, st, E_d, F_d, W_d, beta_d, nullptr, nullptr, true);
    return predict_body(h, N, pos_d, Z_d, cell_h, pbc_h, 0, 1, st, E_d, F_d, W_d, beta_d, nullptr, nullptr, true);
}

extern "C" __attribute__((visibility("default"))) int sgpr_predict(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                            const int32_t* pbc_h, int32_t rank, int32_t world, void* stream, double* E_d, double* F_d,
                            double* W_d, double* beta_d, uint8_t* owned_d) {
    return predict_impl(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, F_d, W_d, beta_d, owned_d, nullptr,
                        h && h->async_mode);
}

// Asynchronous mode of the device-pointer entry points (sgpr_predict, sgpr_predict_p2p): once a sizing step of the same
// shape has run, later steps enqueue their whole kernel sequence without any device-to-host copy or synchronisation.
// The price: a step whose pair list outgrew the capacity (or that met an unknown species) cannot report it from the
// call that enqueued it -- sgpr_check() does, after the caller synchronised the stream.
extern "C" __attribute__((visibility("default"))) int sgpr_set_async(sgpr_handle h, int32_t on) {
    if (!h) {
        set_error("null handle");
        return SGPR_ERR_INVALID;
    }
    h->async_mode = on != 0;
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_check(sgpr_handle h, int64_t* n_pairs_out) {
    if (!h) {
        set_error("null handle");
        return SGPR_ERR_INVALID;
    }
    SGPR_CUDA(cudaSetDevice(h->device));
    long long st[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (h->status_d.p) SGPR_CUDA(cudaMemcpy(st, h->status_d.p, sizeof(st), cudaMemcpyDeviceToHost));
    if (n_pairs_out) *n_pairs_out = h->step_was_warm ? st[0] : h->stats.n_pairs;
    if (h->step_was_warm) h->stats.n_pairs = st[0];
    if (st[1] != h->bad_steps_seen) {
        const long long n_bad = st[1] - h->bad_steps_seen;
        h->bad_steps_seen = st[1];
        h->warm_ok = false;   // the next step sizes its buffers again
        if (st[2] == 1)
            set_error("%lld asynchronous step(s) invalid: atomic number %lld is not in the handle's species table", n_bad, st[3]);
        else if (st[2] == 2)
            set_error("%lld asynchronous step(s) invalid: an atom lies more than 120 cells outside the unit cell", n_bad);
        else
            set_error("%lld asynchronous step(s) invalid: %lld neighbour pairs exceed the capacity %lld sized by an earlier step; "
                      "repeat the step (it will size its buffers again)", n_bad, st[4], st[5]);
        return st[2] == 1 ? SGPR_ERR_SPECIES : st[2] == 2 ? SGPR_ERR_GEOMETRY : SGPR_ERR_RETRY;
    }
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_predict_p2p(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                                const double* cell_h, const int32_t* pbc_h, int32_t rank, int32_t world, void* stream,
                                const uint64_t* peer_f_h, double* E_d, double* W_d) {
    if (!peer_f_h || world < 1) {
        set_error("null peer table");
        return SGPR_ERR_INVALID;
    }
    if (world == 1) {
        set_error("sgpr_predict_p2p needs world > 1 (use sgpr_predict)");
        return SGPR_ERR_INVALID;
    }
    return predict_impl(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, nullptr, W_d, nullptr, nullptr, peer_f_h,
                        h && h->async_mode);
}

// One call per step and rank: clear the next accumulation buffer, evaluate the owned environments (forces on atoms of
// other ranks go straight into their buffers over NVLink), publish E + virial to every peer's mailbox with a stamped
// flag, wait for all peers' flags (= every force kernel has finished), reduce in rank order, collect the own forces.
extern "C" __attribute__((visibility("default"))) int sgpr_p2p_step(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                                                                    const double* cell_h, const int32_t* pbc_h, int32_t rank,
                                                                    int32_t world, void* stream, const uint64_t* peer_base_h,
                                                                    double* E_d, double* F_d, double* W_d, uint8_t* owned_d) {
    if (!h || !peer_base_h || !F_d || !E_d || !W_d || world < 2 || world > SGPR_MAX_RANKS || rank < 0 || rank >= world) {
        set_error("sgpr_p2p_step: bad argument (2 <= world <= %d)", SGPR_MAX_RANKS);
        return SGPR_ERR_INVALID;
    }
    const size_t stride = 3 * (size_t)N + 8;                 // doubles per accumulation buffer
    uint64_t peer_f[SGPR_MAX_RANKS];
    P2PStep px{};
    for (int r = 0; r < world; ++r) {
        peer_f[r] = peer_base_h[r];                          // buffer 0; the step parity is applied on the device
        px.peers.mail[r] = reinterpret_cast<double*>((uintptr_t)(peer_base_h[r] + sizeof(double) * 2 * stride));
    }
    px.own_base = reinterpret_cast<double*>((uintptr_t)peer_base_h[rank]);
    px.stride = (long long)stride;
    px.F_d = F_d;
    px.owned_d = owned_d;
    return predict_impl(h, N, pos_d, Z_d, cell_h, pbc_h, rank, world, stream, E_d, nullptr, W_d, nullptr, nullptr, peer_f,
                        h->async_mode, &px);
}

extern "C" __attribute__((visibility("default"))) int sgpr_p2p_collect(sgpr_handle h, void* stream, const double* own_f_d, double* F_d, uint8_t* owned_d) {
    if (!h || !own_f_d || !F_d) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    const int64_t N = h->last_N;
    if (N > 0)
        scatter_forces_kernel<<<(int)((N + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(), own_f_d,
                                                                      h->owned.as<unsigned char>(), F_d, owned_d);
    SGPR_CUDA(cudaGetLastError());
    return SGPR_OK;
}

static int ensure_pinned(sgpr_context* h, size_t bytes) {
    if (bytes <= h->pinned_bytes) return SGPR_OK;
    // (i8_probs_pinned is an independent fixed-size allocation owned by i8gemm.cu: not touched here)
    if (h->pinned) {
        SGPR_CUDA(cudaStreamSynchronize(h->own_stream));   // no copy may still read the old staging area
        cudaFreeHost(h->pinned);
    }
    h->pinned = nullptr;
    h->pinned_bytes = 0;
    SGPR_CUDA(cudaMallocHost(&h->pinned, bytes + bytes / 4));
    h->pinned_bytes = bytes + bytes / 4;
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_predict_host(sgpr_handle h, int64_t N, const double* pos_h, const int32_t* Z_h,
                                 const double* cell_h, const int32_t* pbc_h, int32_t rank, int32_t world, double* E_h,
                                 double* F_h, double* W_h, double* beta_h, uint8_t* owned_h) {
    if (!h || !E_h || !F_h || !W_h || (N > 0 && (!pos_h || !Z_h))) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    SGPR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->own_stream;
    const size_t nb_pos = sizeof(double) * 3 * (size_t)N, nb_z = sizeof(int32_t) * (size_t)N;
    const size_t nb_out = sizeof(double) * ((beta_h ? 4 : 3) * (size_t)N + 16);
    SGPR_TRY(ensure_pinned(h, nb_pos + nb_z + nb_out + (size_t)N + 64));
    char* pin = (char*)h->pinned;
    double* pin_pos = (double*)pin;
    double* pin_out = (double*)(pin + nb_pos);
    int32_t* pin_z = (int32_t*)(pin + nb_pos + nb_out);
    uint8_t* pin_own = (uint8_t*)(pin + nb_pos + nb_out + nb_z);
    SGPR_TRY(h->stage_pos.ensure(nb_pos + 8));
    SGPR_TRY(h->stage_z.ensure(nb_z + 8));
    SGPR_TRY(h->stage_out.ensure(nb_out + (size_t)N + 64));
    // page-locked caller buffers are copied by the DMA engine directly; pageable ones go through the
    // handle's pinned staging area (one host memcpy each way)
    const bool pos_pinned = N > 0 && is_pinned_host(pos_h), z_pinned = N > 0 && is_pinned_host(Z_h);
    const bool f_pinned = N > 0 && is_pinned_host(F_h);
    if (!pos_pinned) memcpy(pin_pos, pos_h, nb_pos);
    if (!z_pinned) memcpy(pin_z, Z_h, nb_z);
    SGPR_CUDA(cudaMemcpyAsync(h->stage_pos.p, pos_pinned ? pos_h : pin_pos, nb_pos, cudaMemcpyHostToDevice, st));
    SGPR_CUDA(cudaMemcpyAsync(h->stage_z.p, z_pinned ? (const void*)Z_h : (const void*)pin_z, nb_z, cudaMemcpyHostToDevice, st));
    double* out_d = h->stage_out.as<double>();  // [E(1) pad(6) W(9) F(3N) beta(N)]
    double* beta_d = beta_h ? out_d + 16 + 3 * (size_t)N : nullptr;
    uint8_t* own_d = owned_h ? (uint8_t*)(out_d + 16 + (beta_h ? 4 : 3) * (size_t)N) : nullptr;
    // The step runs without any host synchronisation when an earlier step of the same shape sized the buffers; its
    // status block arrives with the results.  An invalid step (pair list outgrew the capacity) is simply repeated
    // as a sizing step: the caller always gets exact results or an error from THIS call.
    for (int attempt = 0; attempt < 2; ++attempt) {
        SGPR_TRY(predict_impl(h, N, h->stage_pos.as<double>(), h->stage_z.as<int32_t>(), cell_h, pbc_h, rank, world, st, out_d,
                              out_d + 16, out_d + 7, beta_d, own_d, nullptr, /*allow_warm=*/attempt == 0));
        if (f_pinned) {
            SGPR_CUDA(cudaMemcpyAsync(pin_out, out_d, sizeof(double) * 16, cudaMemcpyDeviceToHost, st));
            SGPR_CUDA(cudaMemcpyAsync(F_h, out_d + 16, nb_pos, cudaMemcpyDeviceToHost, st));
            if (beta_h)
                SGPR_CUDA(cudaMemcpyAsync(pin_out + 16 + 3 * (size_t)N, beta_d, sizeof(double) * (size_t)N, cudaMemcpyDeviceToHost, st));
        } else {
            SGPR_CUDA(cudaMemcpyAsync(pin_out, out_d, nb_out, cudaMemcpyDeviceToHost, st));
        }
        if (owned_h) SGPR_CUDA(cudaMemcpyAsync(pin_own, own_d, (size_t)N, cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaStreamSynchronize(st));
        if (!h->step_was_warm) break;
        h->stats.n_pairs = h->status_pinned[0];
        if (h->status_pinned[6] == 0) break;
        h->bad_steps_seen = h->status_pinned[1];
        h->warm_ok = false;
    }
    E_h[0] = pin_out[0];
    memcpy(W_h, pin_out + 7, sizeof(double) * 9);
    if (!f_pinned) memcpy(F_h, pin_out + 16, nb_pos);
    if (owned_h) memcpy(owned_h, pin_own, (size_t)N);
    if (beta_h) memcpy(beta_h, pin_out + 16 + 3 * (size_t)N, sizeof(double) * (size_t)N);
    return SGPR_OK;
}

// Atom offsets of a batch of B structures: first_h[0] = 0 and non-decreasing; *N = first_h[B], the batch's atom count.
static int check_batch_first(int B, const int64_t* first_h, int64_t* N) {
    if (first_h[0] != 0) {
        set_error("first_h[0] = %lld, must be 0", (long long)first_h[0]);
        return SGPR_ERR_INVALID;
    }
    for (int b = 0; b < B; ++b)
        if (first_h[b + 1] < first_h[b]) {
            set_error("first_h is not monotone at structure %d (%lld > %lld)", b, (long long)first_h[b], (long long)first_h[b + 1]);
            return SGPR_ERR_INVALID;
        }
    *N = first_h[B];
    if (*N > 0x7fffff00ll) {
        set_error("bad atom count");
        return SGPR_ERR_INVALID;
    }
    return SGPR_OK;
}

// Front end of the batched entry points, from the state reset to the descriptors of the batch's N atoms: per-structure
// geometry, batched cell sort and neighbour list, descriptors; fills bg.  i8: the step may use the int8 GEMM engine
// (when the handle does).  B == 0 stops after the state reset: the caller has nothing more to do.
static int batch_front(sgpr_context* h, int B, const int64_t* first_h, int64_t N, const double* pos_d, const int32_t* Z_d,
                       const double* cell_h, const int32_t* pbc_h, cudaStream_t st, bool i8, bool with_k8, BatchGeom* bg) {
    h->fwd_valid = false;   // no state for sgpr_kernel_backward / sgpr_kernel_jacobian
    h->warm_ok = false;     // the next single-structure step sizes its buffers again
    h->step_was_warm = false;
    if (B == 0) return SGPR_OK;
    h->use_i8_now = i8 && h->use_i8;
    h->stats.i8_ops = 0.0;
    h->stats.gemm_flops = 0.0;
    h->stats.covloss_flops = 0.0;
    h->stats.kernel_launches = 0;
    h->stats.n_atoms = N;
    h->last_N = N;
    // geometry of every structure, as build_geometry gives it alone; bins of the batch one after the other
    std::vector<Geom> gs;
    SGPR_TRY(build_geometry_batch(h, B, first_h, pos_d, cell_h, pbc_h, st, &gs));
    std::vector<int> bin_base(B + 1, 0);
    std::vector<double> cells(9 * (size_t)B);
    long long ncell = 0;
    for (int b = 0; b < B; ++b) {
        bin_base[b] = (int)ncell;
        ncell += gs[b].ncell;
        for (int q = 0; q < 9; ++q) cells[9 * (size_t)b + q] = gs[b].cell[q];
    }
    if ((ncell + 1) * h->S > 0x7fffffffll) {
        set_error("batch too large: %lld bins", ncell);
        return SGPR_ERR_INVALID;
    }
    bin_base[B] = (int)ncell;
    SGPR_TRY(h->b_geom.ensure(sizeof(Geom) * (size_t)B));
    SGPR_TRY(h->b_first.ensure(sizeof(long long) * ((size_t)B + 1)));
    SGPR_TRY(h->b_bins.ensure(sizeof(int) * ((size_t)B + 1)));
    SGPR_TRY(h->b_cell.ensure(sizeof(double) * 9 * (size_t)B));
    SGPR_TRY(h->b_err.ensure(sizeof(unsigned long long) * 2));
    SGPR_TRY(h->astr.ensure(sizeof(int) * ((size_t)N + 1)));
    SGPR_CUDA(cudaMemcpyAsync(h->b_geom.p, gs.data(), sizeof(Geom) * (size_t)B, cudaMemcpyHostToDevice, st));
    SGPR_CUDA(cudaMemcpyAsync(h->b_first.p, first_h, sizeof(long long) * ((size_t)B + 1), cudaMemcpyHostToDevice, st));
    SGPR_CUDA(cudaMemcpyAsync(h->b_bins.p, bin_base.data(), sizeof(int) * ((size_t)B + 1), cudaMemcpyHostToDevice, st));
    SGPR_CUDA(cudaMemcpyAsync(h->b_cell.p, cells.data(), sizeof(double) * 9 * (size_t)B, cudaMemcpyHostToDevice, st));
    *bg = BatchGeom{};
    bg->B = B;
    bg->ncell = (int)ncell;
    bg->geoms = h->b_geom.as<Geom>();
    bg->first = h->b_first.as<long long>();
    bg->bin_base = h->b_bins.as<int>();
    bg->cells = h->b_cell.as<double>();
    bg->astr = h->astr.as<int>();
    bg->err = h->b_err.as<unsigned long long>();
    const Geom unused{};
    // cell sort -> neighbour list (the call's one sizing synchronisation) -> descriptors
    if (h->timing) cudaEventRecord(h->ev[0], st);
    SGPR_TRY(batch_cell_sort(h, N, pos_d, Z_d, *bg, st));
    int64_t n_pairs = 0;
    SGPR_TRY(batch_neighbor_build(h, N, *bg, st, &n_pairs));
    h->stats.n_active = h->n_active;
    h->stats.n_pairs = n_pairs;
    if (h->timing) cudaEventRecord(h->ev[1], st);
    SGPR_TRY(h->phat.ensure(sizeof(double) * ((size_t)N + 1) * h->dp.ldp));
    if (h->use_i8_now) SGPR_TRY(i8_ensure_step_buffers(h, (size_t)N, with_k8));
    SGPR_TRY(descriptor_forward_atoms(h, unused, st, bg));
    if (h->timing) cudaEventRecord(h->ev[2], st);
    return SGPR_OK;
}

// B independent structures in one call (include/sgpr_b200.h).  Same stages as a sizing step of sgpr_predict over the
// concatenated atoms; what differs is per-structure geometry (batched cell sort, neighbour search and image shifts) and
// the per-structure reductions.  The rows are ordinary descriptor rows: GEMMs, covloss and force scatter are shared.
extern "C" __attribute__((visibility("default"))) int sgpr_predict_batch(sgpr_handle h, int32_t B, const int64_t* first_h,
                                                                         const double* pos_d, const int32_t* Z_d,
                                                                         const double* cell_h, const int32_t* pbc_h,
                                                                         void* stream, double* E_d, double* F_d,
                                                                         double* W_d, double* beta_d) {
    if (!h || B < 0 || !first_h || (B > 0 && (!cell_h || !pbc_h || !E_d || !W_d))) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    int64_t N = 0;
    SGPR_TRY(check_batch_first(B, first_h, &N));
    if (N > 0 && (!pos_d || !Z_d || !F_d)) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    if (beta_d && !h->has_choli) {
        set_error("covloss requested but the model has no choli");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    BatchGeom bg;
    SGPR_TRY(batch_front(h, B, first_h, N, pos_d, Z_d, cell_h, pbc_h, st, /*i8=*/true, /*with_k8=*/beta_d != nullptr, &bg));
    if (B == 0) return SGPR_OK;
    const Geom unused{};
    const size_t nrows = (size_t)N + 1;
    if (h->use_i8_now) SGPR_TRY(i8_setup_step(h, st));
    int max_part = 1;
    const RowSpecies rs = row_species(h, &max_part);
    SGPR_TRY(h->erow_part.ensure(sizeof(double) * (size_t)max_part * nrows));
    SGPR_TRY(h->erow.ensure(sizeof(double) * nrows));
    if (!h->use_i8_now) SGPR_TRY(h->gmat.ensure(sizeof(double) * nrows * h->ldg));
    SGPR_TRY(h->gvec.ensure(sizeof(double) * nrows * h->dp.ldp));
    SGPR_TRY(h->epart.ensure(sizeof(double) * kRowEnergyGrid));
    SGPR_TRY(h->fcell.ensure(sizeof(double) * 3 * nrows));
    SGPR_TRY(h->wenv.ensure(sizeof(double) * 9 * nrows));
    SGPR_CUDA(cudaMemsetAsync(h->fcell.p, 0, sizeof(double) * 3 * nrows, st));
    SGPR_CUDA(cudaMemsetAsync(h->wenv.p, 0, sizeof(double) * 9 * nrows, st));
    if (beta_d && !h->use_i8_now) SGPR_TRY(h->kcmat.ensure(sizeof(double) * nrows * h->ldg));
    SGPR_TRY(gemm_stage(h, st, rs, beta_d != nullptr));
    {
        NvtxRange force_range("sgpr:force");
        SGPR_TRY(descriptor_backward_atoms(h, unused, nullptr, st, nullptr, &bg));
        if (N > 0)
            scatter_forces_kernel<<<(int)((N + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(), h->fcell.as<double>(),
                                                                          nullptr, F_d, nullptr);
        batch_reduce_kernel<<<(B + 7) / 8, 256, 0, st>>>(B, bg.first, h->atoms.as<AtomRec>(), h->rowof.as<int>() + (N + 1),
                                                        h->nl_first.as<long long>(), h->erow.as<double>(),
                                                        h->mean_w_d.as<double>(), h->lone_mu.as<double>(),
                                                        h->wenv.as<double>(), E_d, W_d);
        h->stats.kernel_launches += 2;
        SGPR_CUDA(cudaGetLastError());
    }
    if (h->timing) cudaEventRecord(h->ev[4], st);
    if (beta_d) SGPR_TRY(covloss_stage(h, st, N, nullptr, nullptr, beta_d));
    if (h->timing) SGPR_TRY(read_stage_times(h, st));
    return SGPR_OK;
}

// K [N, M] of the N atoms of the last front end into K (caller's rows and columns, lone-lone term included), FP64 GEMM
static int kernel_matrix_caller_order(sgpr_context* h, int64_t N, cudaStream_t st, double* K) {
    SGPR_TRY(h->gmat.ensure(sizeof(double) * ((size_t)N + 1) * h->ldg));
    {
        int max_part = 1;
        for (int s = 0; s < h->S; ++s) max_part = std::max(max_part, gemm_energy_parts(h->m_first[s + 1] - h->m_first[s]));
        SGPR_TRY(h->erow_part.ensure(sizeof(double) * (size_t)max_part * ((size_t)N + 1)));
    }
    SGPR_TRY(h->rowmap.ensure(sizeof(int) * ((size_t)N + 1)));
    SGPR_CUDA(cudaMemsetAsync(K, 0, sizeof(double) * (size_t)N * h->M, st));
    if (N > 0 && h->M > 0) {
        row_to_orig_kernel<<<(int)((N + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(),
                                                                   h->rowof.as<int>() + (N + 1), h->rowmap.as<int>());
        SGPR_TRY(gemm_kernel_matrix(h, K, h->M, h->rowmap.as<int>(), false, st));
        // lone-lone term, in the caller's inducing order
        bool any = false;
        for (int p = 0; p < h->M; ++p) any |= h->ind_lone[p] != 0;
        if (any) {
            lone_k_kernel<<<h->sm_count, 128, 0, st>>>((int)h->n_active, nullptr, h->atoms.as<AtomRec>(),
                                                       h->nl_first.as<long long>(), h->M, h->ind_sp_d.as<int>(),
                                                       h->ind_lone_d.as<unsigned char>(), K, h->lone_w);
        }
        h->stats.kernel_launches += 2;
    }
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_kernel_forward(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                                   const double* cell_h, const int32_t* pbc_h, void* stream, double* K_d) {
    if (!h || !K_d) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    Geom g;
    SGPR_TRY(stage_front(h, N, pos_d, Z_d, cell_h, pbc_h, st, &g));
    SGPR_TRY(kernel_matrix_caller_order(h, N, st, K_d));
    SGPR_CUDA(cudaGetLastError());
    SGPR_CUDA(cudaStreamSynchronize(st));
    h->fwd_valid = true;
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_kernel_backward(sgpr_handle h, const double* gK_d, void* stream, double* gpos_d, double* gcell_h) {
    // Vector-Jacobian product of the LAST sgpr_kernel_forward:  L = sum_im gK[i,m] K[i,m]
    //   dL/dk[i,m] = gK[i,m] xi k^(xi-1)   -> same pipeline as the prediction with mu_m replaced by gK[i,m]
    //   dL/dxyz = -F ;  dL/dcell[k,:] = sum_pairs S_k g = (cell^-T (W + sum_k x_k (x) F_k))[k,:]
    if (!h || !gK_d || !gpos_d || !gcell_h) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    if (!h->fwd_valid) {
        set_error("sgpr_kernel_backward needs a preceding sgpr_kernel_forward on this handle");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    const int64_t N = h->last_N;
    const Geom g = h->last_geom;
    const size_t nrows = (size_t)h->n_active + 1;
    const int nblk_b = backward_grid(h), grid_e = 128, nblk_x = 64;
    h->use_i8_now = false;   // the VJP runs the FP64 GEMM (row_species() reads this)
    int max_part = 1;
    const RowSpecies rs = row_species(h, &max_part);
    SGPR_TRY(h->gmat.ensure(sizeof(double) * nrows * h->ldg));
    SGPR_TRY(h->gvec.ensure(sizeof(double) * nrows * h->dp.ldp));
    SGPR_TRY(h->erow_part.ensure(sizeof(double) * (size_t)max_part * nrows));
    SGPR_TRY(h->erow.ensure(sizeof(double) * nrows));
    SGPR_TRY(h->epart.ensure(sizeof(double) * (grid_e + 16 + 9 * nblk_x)));
    SGPR_TRY(h->wpart.ensure(sizeof(double) * 9 * nblk_b));
    SGPR_TRY(h->fcell.ensure(sizeof(double) * 3 * ((size_t)N + 1)));
    SGPR_CUDA(cudaMemsetAsync(h->wpart.p, 0, sizeof(double) * 9 * nblk_b, st));
    SGPR_CUDA(cudaMemsetAsync(h->fcell.p, 0, sizeof(double) * 3 * ((size_t)N + 1), st));
    SGPR_CUDA(cudaMemsetAsync(h->epart.p, 0, sizeof(double) * (grid_e + 16 + 9 * nblk_x), st));
    if (N > 0 && h->M > 0) {
        SGPR_TRY(gemm_kernel_matrix(h, nullptr, h->M, h->rowmap.as<int>(), false, st, gK_d));
        row_energy_kernel<<<grid_e, 256, 0, st>>>((int)h->n_active, rs, h->row_first_d.as<int>(), h->erow_part.as<double>(),
                                                  (int)nrows, nullptr, h->erow.as<double>(), h->epart.as<double>());
        SGPR_TRY(gemm_back_projection(h, st));
        SGPR_TRY(descriptor_backward_atoms(h, g, nullptr, st));
    }
    double* xf_part = h->epart.as<double>() + grid_e + 16;
    double* EW = h->epart.as<double>() + grid_e;   // [E, W(9)] scratch
    if (N > 0)
        vjp_finish_kernel<<<nblk_x, 128, 0, st>>>(N, h->atoms.as<AtomRec>(), h->fcell.as<double>(), gpos_d, xf_part);
    final_reduce_kernel<<<1, 320, 0, st>>>(0, nullptr, 0, nullptr, nblk_b, h->wpart.as<double>(), EW, EW + 1);
    double host[16 + 9 * 64];
    SGPR_CUDA(cudaMemcpyAsync(host, EW, sizeof(double) * (16 + 9 * nblk_x), cudaMemcpyDeviceToHost, st));
    SGPR_CUDA(cudaStreamSynchronize(st));
    double Y[9];
    for (int q = 0; q < 9; ++q) {
        double xf = 0.0;
        for (int b = 0; b < nblk_x; ++b) xf += host[16 + b * 9 + q];
        Y[q] = host[1 + q] + xf;   // W + sum x (x) F = cell^T (sum_pairs S (x) g)
    }
    // C = cell^-T Y ;  g.inv = cell^-1 (frac_c = sum_k pos_k inv[k][c])  ->  C[k][b] = sum_a inv[a][k] Y[a][b]
    for (int k = 0; k < 3; ++k)
        for (int b = 0; b < 3; ++b) {
            double c = 0.0;
            for (int a = 0; a < 3; ++a) c += g.inv[a * 3 + k] * Y[a * 3 + b];
            gcell_h[k * 3 + b] = g.pbc[k] ? c : 0.0;
        }
    SGPR_CUDA(cudaGetLastError());
    return SGPR_OK;
}

// Inducing LCEs m0 <= m < m1 (caller's order) of the Jacobian kernel: sorted positions grouped by central species, then
// their output columns, into h->jsel.  Excluded central species get no entries: their columns stay zero.
static int upload_selection(sgpr_context* h, int m0, int m1, cudaStream_t st, JacTarget* t) {
    std::vector<int> sel, col;
    t->sel_first[0] = 0;
    for (int s = 0; s < SGPR_MAX_SPECIES; ++s) {
        if (s < h->S && h->dp.central_enabled[s])
            for (int p = h->m_first[s]; p < h->m_first[s + 1]; ++p) {
                const int m = h->ind_perm[p];
                if (m >= m0 && m < m1) {
                    sel.push_back(p);
                    col.push_back(m - m0);
                }
            }
        t->sel_first[s + 1] = (int)sel.size();
    }
    t->n_sel = (int)sel.size();
    t->ncol = m1 - m0;
    sel.insert(sel.end(), col.begin(), col.end());
    SGPR_TRY(h->jsel.ensure(sizeof(int) * (sel.size() + 1)));
    if (!sel.empty()) SGPR_CUDA(cudaMemcpyAsync(h->jsel.p, sel.data(), sizeof(int) * sel.size(), cudaMemcpyHostToDevice, st));
    t->sel = h->jsel.as<int>();
    return SGPR_OK;
}

// Jacobian kernel of the last front end's atoms against inducing LCEs m0 <= m < m1 into J_d [ncol, N, 3] and W_d
// [B, ncol, 9], both zeroed here.  cells_d [B, 9]: the structures' cells; astr_d: structure of each cell-order atom
// (nullptr: one structure).
static int jacobian_stage(sgpr_context* h, int m0, int m1, int B, const double* cells_d, const int* astr_d, double* J_d,
                          double* W_d, cudaStream_t st) {
    const int64_t N = h->last_N;
    const int ncol = m1 - m0;
    JacTarget t{};
    SGPR_TRY(upload_selection(h, m0, m1, st, &t));
    t.n_atoms = N;
    t.J = J_d;
    t.W = W_d;
    t.cells = cells_d;
    t.astr = astr_d;
    if (N > 0) SGPR_CUDA(cudaMemsetAsync(J_d, 0, sizeof(double) * 3 * (size_t)N * ncol, st));
    SGPR_CUDA(cudaMemsetAsync(W_d, 0, sizeof(double) * 9 * (size_t)B * ncol, st));
    if (N > 0) SGPR_TRY(descriptor_jacobian_atoms(h, t, st));
    return SGPR_OK;
}

// Training-time kernels of the structure of the LAST sgpr_kernel_forward against inducing LCEs m0 <= m < m1
// (caller's order): the Jacobian of Ke[m] = sum_i K[i,m] for all of them in one launch (descriptor.cu: jacobian_kernel).
extern "C" __attribute__((visibility("default"))) int sgpr_kernel_jacobian(sgpr_handle h, int32_t m0, int32_t m1, void* stream, double* J_d, double* W_d) {
    if (!h || !J_d || !W_d) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    if (!h->fwd_valid) {
        set_error("sgpr_kernel_jacobian needs a preceding sgpr_kernel_forward on this handle");
        return SGPR_ERR_INVALID;
    }
    if (m0 < 0 || m1 > h->M || m0 > m1) {
        set_error("inducing range [%d, %d) outside [0, %d)", m0, m1, h->M);
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    if (m1 == m0) return SGPR_OK;
    h->use_i8_now = false;
    SGPR_TRY(h->b_cell.ensure(sizeof(double) * 9));
    SGPR_CUDA(cudaMemcpyAsync(h->b_cell.p, h->last_geom.cell, sizeof(double) * 9, cudaMemcpyHostToDevice, st));
    SGPR_TRY(jacobian_stage(h, m0, m1, 1, h->b_cell.as<double>(), nullptr, J_d, W_d, st));
    SGPR_CUDA(cudaGetLastError());
    SGPR_CUDA(cudaStreamSynchronize(st));
    return SGPR_OK;
}

// Training-time kernels of B independent structures in one call (include/sgpr_b200.h): the front end of
// sgpr_predict_batch, the kernel matrix into a scratch buffer, per-structure column sums (Ke) and the Jacobian kernel.
extern "C" __attribute__((visibility("default"))) int sgpr_kernel_jacobian_batch(sgpr_handle h, int32_t B, const int64_t* first_h,
                                                                                 const double* pos_d, const int32_t* Z_d,
                                                                                 const double* cell_h, const int32_t* pbc_h,
                                                                                 int32_t m0, int32_t m1, void* stream,
                                                                                 double* Ke_d, double* J_d, double* W_d) {
    if (!h || B < 0 || !first_h || (B > 0 && (!cell_h || !pbc_h || !Ke_d))) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    if ((J_d == nullptr) != (W_d == nullptr)) {
        set_error("J_d and W_d must both be given (Jacobian) or both be NULL (Ke only)");
        return SGPR_ERR_INVALID;
    }
    if (m0 < 0 || m1 > h->M || m0 > m1) {
        set_error("inducing range [%d, %d) outside [0, %d)", m0, m1, h->M);
        return SGPR_ERR_INVALID;
    }
    int64_t N = 0;
    SGPR_TRY(check_batch_first(B, first_h, &N));
    if (N > 0 && (!pos_d || !Z_d)) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    BatchGeom bg;
    SGPR_TRY(batch_front(h, B, first_h, N, pos_d, Z_d, cell_h, pbc_h, st, /*i8=*/false, /*with_k8=*/false, &bg));
    if (B == 0) return SGPR_OK;
    const int ncol = m1 - m0;
    // K [N, M] (caller's rows and columns, lone-lone term included) -> Ke
    SGPR_TRY(h->kscr.ensure(sizeof(double) * ((size_t)N * h->M + 1)));
    double* K = h->kscr.as<double>();
    SGPR_TRY(kernel_matrix_caller_order(h, N, st, K));
    if (ncol > 0) {
        const long long n = (long long)B * ncol;
        ke_reduce_kernel<<<(int)std::min<long long>((n + 255) / 256, (long long)h->sm_count * 16), 256, 0, st>>>(
            B, bg.first, h->M, m0, ncol, K, Ke_d);
        h->stats.kernel_launches += 1;
    }
    if (h->timing) cudaEventRecord(h->ev[3], st);
    if (J_d && ncol > 0) {
        NvtxRange jac_range("sgpr:jacobian");
        SGPR_TRY(jacobian_stage(h, m0, m1, B, bg.cells, bg.astr, J_d, W_d, st));
    }
    SGPR_CUDA(cudaGetLastError());
    if (h->timing) {
        cudaEventRecord(h->ev[4], st);
        SGPR_TRY(read_stage_times(h, st));
        h->stats.ms_beta = 0.0f;
    }
    return SGPR_OK;
}

// =====================================================================================
// parity hooks
// =====================================================================================
extern "C" __attribute__((visibility("default"))) int sgpr_neighbors(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                              const int32_t* pbc_h, void* stream, int64_t* first_d, int32_t* j_d, int8_t* S_d,
                              int64_t capacity, int64_t* nnz_h) {
    if (!h || !first_d || !nnz_h) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    Geom g;
    h->stats.kernel_launches = 0;
    h->last_N = N;
    SGPR_TRY(build_geometry(h, N, pos_d, cell_h, pbc_h, st, &g));
    SGPR_TRY(cell_sort(h, N, pos_d, Z_d, g, st));
    h->active_all = true;
    h->n_active = N;
    int64_t n_pairs = 0;
    SGPR_TRY(neighbor_build(h, N, g, st, &n_pairs));
    *nnz_h = n_pairs;
    // counts in caller order -> exclusive scan -> export
    SGPR_TRY(h->misc.ensure(sizeof(long long) * ((size_t)N + 2)));
    long long* cnt = h->misc.as<long long>();
    nl_count_orig_kernel<<<(int)((N + 1 + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(),
                                                                     h->nl_first.as<long long>(), cnt);
    SGPR_TRY(scan_exclusive_ll(h, cnt, (long long*)first_d, (int)N + 1, st));
    if (n_pairs <= capacity && N > 0 && j_d && S_d) {
        nl_export_kernel<<<(int)((N * 32 + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(), h->nl_pairs.as<PairRec>(),
                                                                      h->nl_first.as<long long>(), (const long long*)first_d,
                                                                      j_d, S_d);
    }
    SGPR_CUDA(cudaGetLastError());
    SGPR_CUDA(cudaStreamSynchronize(st));
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_descriptors(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                                const int32_t* pbc_h, void* stream, double* P_d) {
    if (!h || !P_d) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    Geom g;
    SGPR_TRY(stage_front(h, N, pos_d, Z_d, cell_h, pbc_h, st, &g));
    // source row of caller atom i: rowof[cell index of i]
    SGPR_TRY(h->rowmap.ensure(sizeof(int) * 2 * ((size_t)N + 1)));
    if (N > 0) {
        orig_to_row_kernel<<<(int)((N + 255) / 256), 256, 0, st>>>(N, h->atoms.as<AtomRec>(),
                                                                   h->rowof.as<int>() + (N + 1), h->rowmap.as<int>());
        SGPR_TRY(unpack_descriptors(h, N, h->phat.as<double>(), h->rowmap.as<int>(), P_d, st));
    }
    SGPR_CUDA(cudaGetLastError());
    SGPR_CUDA(cudaStreamSynchronize(st));
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_inducing_descriptors(sgpr_handle h, void* stream, double* Zhat_d) {
    if (!h || !Zhat_d) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    if (h->M == 0) return SGPR_OK;
    // source row of caller's inducing m = its sorted position
    std::vector<int> src(h->M);
    for (int p = 0; p < h->M; ++p) src[h->ind_perm[p]] = p;
    SGPR_TRY(h->rowmap.ensure(sizeof(int) * ((size_t)h->M + 1)));
    SGPR_CUDA(cudaMemcpyAsync(h->rowmap.p, src.data(), sizeof(int) * h->M, cudaMemcpyHostToDevice, st));
    SGPR_CUDA(cudaStreamSynchronize(st));
    SGPR_TRY(unpack_descriptors(h, h->M, h->zhat.as<double>(), h->rowmap.as<int>(), Zhat_d, st));
    SGPR_CUDA(cudaStreamSynchronize(st));
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_kernel_envs(sgpr_handle h, int32_t n_env, const int32_t* env_Z_h,
                                                                       const int64_t* env_first_h, const double* env_r_h,
                                                                       const int32_t* env_b_h, void* stream, double* K_d,
                                                                       double* P_d) {
    if (!h || n_env < 0 || (n_env > 0 && (!env_Z_h || !env_first_h)) || (!K_d && !P_d)) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SGPR_CUDA(cudaSetDevice(h->device));
    if (n_env == 0) return SGPR_OK;
    const DescParams& dp = h->dp;
    const int64_t nnz = env_first_h[n_env] - env_first_h[0];
    if (nnz < 0 || (nnz > 0 && (!env_r_h || !env_b_h))) {
        set_error("bad CSR of the environments");
        return SGPR_ERR_INVALID;
    }
    std::vector<int> sp(n_env), rows(n_env);
    std::vector<unsigned char> lone(n_env), esp((size_t)nnz + 1);
    std::vector<long long> first(n_env + 1);
    for (int e = 0; e < n_env; ++e) {
        const int z = env_Z_h[e];
        if (z < 0 || z >= 128 || h->z_to_species[z] < 0) {
            set_error("environment %d: species Z=%d not in the species table", e, z);
            return SGPR_ERR_SPECIES;
        }
        sp[e] = h->z_to_species[z];
        rows[e] = e;
        first[e] = env_first_h[e] - env_first_h[0];
        lone[e] = env_first_h[e + 1] == env_first_h[e];
    }
    first[n_env] = nnz;
    const int64_t o = env_first_h[0];
    for (int64_t k = 0; k < nnz; ++k) {
        const int z = env_b_h[o + k];
        if (z < 0 || z >= 128 || h->z_to_species[z] < 0) {
            set_error("environment neighbour species Z=%d not in the species table", z);
            return SGPR_ERR_SPECIES;
        }
        esp[k] = (unsigned char)h->z_to_species[z];
    }
    DevBuf b_first, b_r, b_sp, b_row, b_p, b_esp, b_lone, b_ipsp, b_iplone, b_en;
    int stt = SGPR_OK;
    auto done = [&](int code) {
        cudaStreamSynchronize(st);
        for (DevBuf* b : {&b_first, &b_r, &b_sp, &b_row, &b_p, &b_esp, &b_lone, &b_ipsp, &b_iplone, &b_en}) b->release();
        return code;
    };
#define ENVS_TRY(x)                      \
    do {                                 \
        stt = (x);                       \
        if (stt != SGPR_OK) return done(stt); \
    } while (0)
    ENVS_TRY(upload(b_first, first.data(), sizeof(long long) * (n_env + 1)));
    ENVS_TRY(upload(b_r, env_r_h ? env_r_h + 3 * o : nullptr, sizeof(double) * 3 * nnz));
    ENVS_TRY(upload(b_sp, esp.data(), (size_t)nnz));
    ENVS_TRY(upload(b_row, rows.data(), sizeof(int) * n_env));
    ENVS_TRY(b_p.ensure(sizeof(double) * ((size_t)n_env + 1) * dp.ldp));
    if (cudaMemsetAsync(b_p.p, 0, sizeof(double) * ((size_t)n_env + 1) * dp.ldp, st) != cudaSuccess) return done(SGPR_ERR_CUDA);
    ENVS_TRY(descriptor_forward_env(h, n_env, b_first.as<long long>(), b_r.as<double>(), b_sp.as<unsigned char>(),
                                    b_row.as<int>(), b_p.as<double>(), st));
    if (K_d && h->M > 0) {
        ENVS_TRY(upload(b_esp, sp.data(), sizeof(int) * n_env));
        ENVS_TRY(upload(b_lone, lone.data(), (size_t)n_env));
        ENVS_TRY(upload(b_ipsp, h->ind_sp.data(), sizeof(int) * h->M));
        ENVS_TRY(upload(b_iplone, h->ind_lone.data(), (size_t)h->M));
        ENVS_TRY(upload(b_en, dp.central_enabled, sizeof(int) * SGPR_MAX_SPECIES));
        env_kernel_rows_kernel<<<n_env, 256, 0, st>>>(n_env, h->M, dp.D, dp.ldp, b_p.as<double>(), h->zhat.as<double>(),
                                                      b_esp.as<int>(), b_lone.as<unsigned char>(), h->ind_perm_d.as<int>(),
                                                      b_ipsp.as<int>(), b_iplone.as<unsigned char>(), b_en.as<int>(), h->xi,
                                                      h->xi_int, h->lone_w, K_d);
        h->stats.kernel_launches += 1;
    }
    if (P_d) ENVS_TRY(unpack_descriptors(h, n_env, b_p.as<double>(), nullptr, P_d, st));
#undef ENVS_TRY
    if (cudaGetLastError() != cudaSuccess) {
        set_error("sgpr_kernel_envs: kernel launch failed");
        return done(SGPR_ERR_CUDA);
    }
    return done(SGPR_OK);
}

extern "C" __attribute__((visibility("default"))) int sgpr_get_stats(sgpr_handle h, sgpr_stats* out) {
    if (!h || !out) {
        set_error("null argument");
        return SGPR_ERR_INVALID;
    }
    *out = h->stats;
    return SGPR_OK;
}

extern "C" __attribute__((visibility("default"))) int sgpr_enable_timing(sgpr_handle h, int32_t on) {
    if (!h) {
        set_error("null handle");
        return SGPR_ERR_INVALID;
    }
    h->timing = on != 0;
    return SGPR_OK;
}
