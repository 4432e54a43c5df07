// Cell-list neighbour search (SURVEY.md section 8 rows a1, a2).
//
// Semantics restated from the reference's call site descriptor/atoms.py:348-368
// (ASE NeighborList(N*[rc/2], skin=0, self_interaction=False, bothways=True)):
//   pair (i, j, S) kept  iff  sqrt(|x_j - x_i + S.cell|^2) < rc  (strict), both
//   directions, (i == j, S == 0) dropped, periodic images of the same atom kept,
//   S relative to the positions as given.
// The distance is evaluated from the caller's (unwrapped) positions in the reference's
// operation order (r = (x_j - x_i) + sum_k S_k cell_k, no FMA contraction), so the
// accept/reject decision is the same floating-point comparison the reference makes.
// (Candidates farther from the cutoff sphere than the rounding error of a float test on
// bin-relative coordinates are decided by that test; see neighbor_bin_kernel.)
//
// Layout: atoms are counting-sorted by key = bin*S + species ("cell order"); a bin's
// atoms are one contiguous run, ordered by species then by original index
// (deterministic).  Descriptor rows use a second, species-major order ("row order") so
// that the kernel GEMM sees one contiguous row block per central species.
#include <cub/device/device_scan.cuh>
#include <math.h>

#include "sgpr_internal.cuh"

namespace sgpr {

// ---------------------------------------------------------------------------------
// geometry (host)
// ---------------------------------------------------------------------------------
static void cross3(const double* a, const double* b, double* c) {
    c[0] = a[1] * b[2] - a[2] * b[1];
    c[1] = a[2] * b[0] - a[0] * b[2];
    c[2] = a[0] * b[1] - a[1] * b[0];
}
static double norm3(const double* a) { return sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); }

// Replace zero lattice vectors by unit vectors orthogonal to the others (what ASE's
// Atoms.get_cell(complete=True) hands to the neighbour list).
static void complete_cell(double* c) {
    bool missing[3];
    int nmiss = 0;
    for (int i = 0; i < 3; ++i) {
        missing[i] = (c[3 * i] == 0.0 && c[3 * i + 1] == 0.0 && c[3 * i + 2] == 0.0);
        nmiss += missing[i];
    }
    if (nmiss == 3) {
        for (int i = 0; i < 9; ++i) c[i] = (i % 4 == 0) ? 1.0 : 0.0;
    } else if (nmiss == 2) {
        int p = !missing[0] ? 0 : (!missing[1] ? 1 : 2);
        double v[3] = {c[3 * p], c[3 * p + 1], c[3 * p + 2]};
        double n = norm3(v);
        for (int k = 0; k < 3; ++k) v[k] /= n;
        int m = 0;
        for (int k = 1; k < 3; ++k)
            if (fabs(v[k]) < fabs(v[m])) m = k;
        double t[3] = {0, 0, 0};
        t[m] = 1.0;
        double e1[3], e2[3];
        cross3(v, t, e1);
        n = norm3(e1);
        for (int k = 0; k < 3; ++k) e1[k] /= n;
        cross3(v, e1, e2);
        int q = 0;
        for (int i = 0; i < 3; ++i)
            if (missing[i]) {
                const double* e = (q++ == 0) ? e1 : e2;
                for (int k = 0; k < 3; ++k) c[3 * i + k] = e[k];
            }
    } else if (nmiss == 1) {
        int i = missing[0] ? 0 : (missing[1] ? 1 : 2);
        double e[3];
        cross3(&c[3 * ((i + 1) % 3)], &c[3 * ((i + 2) % 3)], e);
        double n = norm3(e);
        for (int k = 0; k < 3; ++k) c[3 * i + k] = e[k] / n;
    }
}

__global__ void frac_minmax_kernel(int64_t N, const double* __restrict__ pos, Geom g, double* __restrict__ part) {
    // per-block min/max of the fractional coordinates (non-periodic axes need a bounding box)
    __shared__ double smin[3][256], smax[3][256];
    double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        double x = pos[3 * i], y = pos[3 * i + 1], z = pos[3 * i + 2];
        for (int c = 0; c < 3; ++c) {
            double f = x * g.inv[c] + y * g.inv[3 + c] + z * g.inv[6 + c];
            mn[c] = fmin(mn[c], f);
            mx[c] = fmax(mx[c], f);
        }
    }
    for (int c = 0; c < 3; ++c) {
        smin[c][threadIdx.x] = mn[c];
        smax[c][threadIdx.x] = mx[c];
    }
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s)
            for (int c = 0; c < 3; ++c) {
                smin[c][threadIdx.x] = fmin(smin[c][threadIdx.x], smin[c][threadIdx.x + s]);
                smax[c][threadIdx.x] = fmax(smax[c][threadIdx.x], smax[c][threadIdx.x + s]);
            }
        __syncthreads();
    }
    if (threadIdx.x == 0)
        for (int c = 0; c < 3; ++c) {
            part[blockIdx.x * 6 + c] = smin[c][0];
            part[blockIdx.x * 6 + 3 + c] = smax[c][0];
        }
}

// completed cell, its inverse and the distances between opposite faces (host)
static int geom_cell(const double* cell_h, const int32_t* pbc_h, double rc, Geom* g, double* hface) {
    for (int i = 0; i < 9; ++i) g->cell[i] = cell_h[i];
    for (int c = 0; c < 3; ++c) g->pbc[c] = pbc_h[c] ? 1 : 0;
    complete_cell(g->cell);
    const double* a = g->cell;
    double bc[3], ca[3], ab[3];
    cross3(a + 3, a + 6, bc);
    cross3(a + 6, a + 0, ca);
    cross3(a + 0, a + 3, ab);
    double vol = a[0] * bc[0] + a[1] * bc[1] + a[2] * bc[2];
    if (!(fabs(vol) > 1e-12)) {
        set_error("singular cell (volume %g)", vol);
        return SGPR_ERR_GEOMETRY;
    }
    // inverse: columns are the reciprocal vectors b_c = (a_{c+1} x a_{c+2}) / vol
    const double* rec[3] = {bc, ca, ab};
    for (int c = 0; c < 3; ++c)
        for (int k = 0; k < 3; ++k) g->inv[k * 3 + c] = rec[c][k] / vol;
    g->rc = rc;
    for (int c = 0; c < 3; ++c) hface[c] = fabs(vol) / norm3(rec[c]);
    return SGPR_OK;
}

// bins and stencil reach from the fractional bounds lo / hi of the non-periodic axes (host)
static void geom_bins(Geom* g, const double* hface, const double* lo, const double* hi, int64_t N) {
    const double rcs = g->rc * (1.0 + 1e-7);
    for (int c = 0; c < 3; ++c) {
        if (g->pbc[c]) {
            int nb = (int)floor(hface[c] / rcs);
            if (nb < 1) nb = 1;
            g->nb[c] = nb;
            g->reach[c] = (int)ceil(rcs / (hface[c] / nb));
            g->flo[c] = 0.0;
            g->fscale[c] = (double)nb;
        } else {
            double ext = (hi[c] - lo[c]) * hface[c];
            int nb = (int)floor(ext / rcs);
            if (nb < 1) nb = 1;
            g->nb[c] = nb;
            g->reach[c] = 1;
            g->flo[c] = lo[c];
            g->fscale[c] = (hi[c] > lo[c]) ? nb / (hi[c] - lo[c]) : 0.0;
        }
    }
    // keep the cell table small relative to the number of atoms (larger bins stay correct)
    const double limit = fmax(4096.0, 4.0 * (double)N);
    for (;;) {
        double nc = (double)g->nb[0] * g->nb[1] * g->nb[2];
        if (nc <= limit) break;
        int c = 0;
        for (int k = 1; k < 3; ++k)
            if (g->nb[k] > g->nb[c]) c = k;
        int nb = (g->nb[c] + 1) / 2;
        if (g->pbc[c]) {
            g->fscale[c] = (double)nb;
            g->reach[c] = (int)ceil(rcs / (hface[c] / nb));
        } else {
            g->fscale[c] *= (double)nb / g->nb[c];
        }
        g->nb[c] = nb;
    }
    g->ncell = g->nb[0] * g->nb[1] * g->nb[2];
}

int build_geometry(sgpr_context* h, int64_t N, const double* pos_d, const double* cell_h, const int32_t* pbc_h,
                   cudaStream_t st, Geom* g) {
    double hface[3];
    SGPR_TRY(geom_cell(cell_h, pbc_h, h->dp.rc, g, hface));
    bool open = !(g->pbc[0] && g->pbc[1] && g->pbc[2]);
    double lo[3] = {0, 0, 0}, hi[3] = {1, 1, 1};
    if (open && N > 0) {
        int nblk = 64;
        SGPR_TRY(h->misc.ensure(sizeof(double) * 6 * nblk));
        frac_minmax_kernel<<<nblk, 256, 0, st>>>(N, pos_d, *g, h->misc.as<double>());
        std::vector<double> part(6 * nblk);
        SGPR_CUDA(cudaMemcpyAsync(part.data(), h->misc.p, sizeof(double) * 6 * nblk, cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaStreamSynchronize(st));
        for (int c = 0; c < 3; ++c) {
            lo[c] = 1e300;
            hi[c] = -1e300;
            for (int b = 0; b < nblk; ++b) {
                lo[c] = fmin(lo[c], part[b * 6 + c]);
                hi[c] = fmax(hi[c], part[b * 6 + 3 + c]);
            }
        }
    }
    geom_bins(g, hface, lo, hi, N);
    return SGPR_OK;
}

// Bounds of the fractional coordinates of the batch's non-periodic structures: one block per structure (list `which`).
__global__ void batch_minmax_kernel(const int* __restrict__ which, const long long* __restrict__ first,
                                    const double* __restrict__ pos, const Geom* __restrict__ geoms, double* __restrict__ out) {
    __shared__ double smin[3][256], smax[3][256];
    const int b = which[blockIdx.x];
    const Geom& g = geoms[b];
    double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
    for (long long i = first[b] + threadIdx.x; i < first[b + 1]; i += blockDim.x) {
        double x = pos[3 * i], y = pos[3 * i + 1], z = pos[3 * i + 2];
        for (int c = 0; c < 3; ++c) {
            double f = x * g.inv[c] + y * g.inv[3 + c] + z * g.inv[6 + c];
            mn[c] = fmin(mn[c], f);
            mx[c] = fmax(mx[c], f);
        }
    }
    for (int c = 0; c < 3; ++c) {
        smin[c][threadIdx.x] = mn[c];
        smax[c][threadIdx.x] = mx[c];
    }
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s)
            for (int c = 0; c < 3; ++c) {
                smin[c][threadIdx.x] = fmin(smin[c][threadIdx.x], smin[c][threadIdx.x + s]);
                smax[c][threadIdx.x] = fmax(smax[c][threadIdx.x], smax[c][threadIdx.x + s]);
            }
        __syncthreads();
    }
    if (threadIdx.x == 0)
        for (int c = 0; c < 3; ++c) {
            out[blockIdx.x * 6 + c] = smin[c][0];
            out[blockIdx.x * 6 + 3 + c] = smax[c][0];
        }
}

int build_geometry_batch(sgpr_context* h, int B, const int64_t* first_h, const double* pos_d, const double* cell_h,
                         const int32_t* pbc_h, cudaStream_t st, std::vector<Geom>* gs) {
    gs->assign(B, Geom{});
    std::vector<double> hface(3 * (size_t)B), lohi(6 * (size_t)B);
    std::vector<int> which;
    for (int b = 0; b < B; ++b) {
        const int rc = geom_cell(cell_h + 9 * (size_t)b, pbc_h + 3 * (size_t)b, h->dp.rc, &(*gs)[b], &hface[3 * (size_t)b]);
        if (rc != SGPR_OK) {
            const std::string msg = sgpr_last_error();
            set_error("structure %d: %s", b, msg.c_str());
            return rc;
        }
        for (int c = 0; c < 3; ++c) {
            lohi[6 * (size_t)b + c] = 0.0;
            lohi[6 * (size_t)b + 3 + c] = 1.0;
        }
        const Geom& g = (*gs)[b];
        if (!(g.pbc[0] && g.pbc[1] && g.pbc[2]) && first_h[b + 1] > first_h[b]) which.push_back(b);
    }
    if (!which.empty()) {
        const int n = (int)which.size();
        SGPR_TRY(h->b_geom.ensure(sizeof(Geom) * (size_t)B));
        SGPR_TRY(h->b_first.ensure(sizeof(long long) * ((size_t)B + 1)));
        SGPR_TRY(h->b_bins.ensure(sizeof(int) * ((size_t)B + 1)));
        SGPR_TRY(h->misc.ensure(sizeof(double) * 6 * (size_t)n));
        SGPR_CUDA(cudaMemcpyAsync(h->b_geom.p, gs->data(), sizeof(Geom) * (size_t)B, cudaMemcpyHostToDevice, st));
        SGPR_CUDA(cudaMemcpyAsync(h->b_first.p, first_h, sizeof(long long) * ((size_t)B + 1), cudaMemcpyHostToDevice, st));
        SGPR_CUDA(cudaMemcpyAsync(h->b_bins.p, which.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
        batch_minmax_kernel<<<n, 256, 0, st>>>(h->b_bins.as<int>(), h->b_first.as<long long>(), pos_d, h->b_geom.as<Geom>(),
                                               h->misc.as<double>());
        SGPR_CUDA(cudaGetLastError());
        std::vector<double> part(6 * (size_t)n);
        SGPR_CUDA(cudaMemcpyAsync(part.data(), h->misc.p, sizeof(double) * 6 * (size_t)n, cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaStreamSynchronize(st));
        for (int k = 0; k < n; ++k)
            for (int q = 0; q < 6; ++q) lohi[6 * (size_t)which[k] + q] = part[6 * (size_t)k + q];
    }
    for (int b = 0; b < B; ++b)
        geom_bins(&(*gs)[b], &hface[3 * (size_t)b], &lohi[6 * (size_t)b], &lohi[6 * (size_t)b + 3], first_h[b + 1] - first_h[b]);
    return SGPR_OK;
}

// ---------------------------------------------------------------------------------
// counting sort into cell order
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void frac_bin(const Geom& g, double x, double y, double z, int* bin3, int* w3) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        double f = x * g.inv[c] + y * g.inv[3 + c] + z * g.inv[6 + c];
        int w = 0;
        if (g.pbc[c]) {
            double fl = floor(f);
            w = (int)fl;
            f -= fl;
        } else {
            f -= g.flo[c];
        }
        int b = (int)(f * g.fscale[c]);
        b = max(0, min(g.nb[c] - 1, b));
        bin3[c] = b;
        w3[c] = w;
    }
}

// the geometry an environment's search uses: the call's, or (batch) that of the centre's structure
template <bool BATCH>
__device__ __forceinline__ const Geom& env_geom(const Geom& g, const BatchGeom& bg, int b) {
    if constexpr (BATCH)
        return bg.geoms[b];
    else
        return g;
}

// structure of atom i (first: atom offsets) or of bin i (first: bin_base): the last b with first[b] <= i (empty
// structures are skipped; every structure has at least one bin)
template <class T>
__device__ __forceinline__ int batch_of(const T* __restrict__ first, int B, long long i) {
    int lo = 0, hi = B;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (first[mid] <= i) lo = mid;
        else hi = mid;
    }
    return lo;
}

// BATCH: keys (bin_base[b] + bin) * S + species -- structure-major, so every structure is one contiguous range of the
// cell order and of each species' rows; errors go to bg.err and name the first failing structure (atomicMin)
template <bool BATCH>
__global__ void bin_count_kernel(int64_t N, const double* __restrict__ pos, const int32_t* __restrict__ Z,
                                 const int* __restrict__ ztab, Geom g_call, int S, int* __restrict__ cnt,
                                 int* __restrict__ key_out, int* __restrict__ rank_out, int* __restrict__ err,
                                 BatchGeom bg = BatchGeom{}) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    int sb = 0, bbase = 0;
    if constexpr (BATCH) {
        sb = batch_of(bg.first, bg.B, i);
        bbase = bg.bin_base[sb];
    }
    const Geom& g = env_geom<BATCH>(g_call, bg, sb);
    int z = Z[i];
    int s = (z >= 0 && z < 128) ? ztab[z] : -1;
    if (s < 0) {
        if constexpr (BATCH) {
            atomicMin(&bg.err[0], ((unsigned long long)sb << 32) | (unsigned)z);
        } else {
            atomicExch(&err[0], 1);
            atomicExch(&err[1], z);
        }
        s = 0;
    }
    int b[3], w[3];
    frac_bin(g, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], b, w);
    if (abs(w[0]) > 120 || abs(w[1]) > 120 || abs(w[2]) > 120) {
        if constexpr (BATCH)
            atomicMin(&bg.err[1], (unsigned long long)sb);
        else
            atomicExch(&err[0], 2);
    }
    int bin = bbase + (b[0] * g.nb[1] + b[1]) * g.nb[2] + b[2];
    int key = bin * S + s;
    key_out[i] = key;
    rank_out[i] = atomicAdd(&cnt[key], 1);
}

__global__ void transpose_cnt_kernel(int ncell, int S, const int* __restrict__ cnt, int* __restrict__ cntT) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= ncell * S) return;
    int bin = k / S, s = k - bin * S;
    cntT[s * ncell + bin] = cnt[k];
}

__global__ void scatter_order_kernel(int64_t N, const int* __restrict__ key, const int* __restrict__ rank,
                                     const int* __restrict__ cstart, int* __restrict__ order) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    order[cstart[key[i]] + rank[i]] = (int)i;
}

// Exclusive prefix sum of n items by ONE block of 1024 threads, in tiles of 8192 with a running carry.  Lanes read
// consecutive items (coalesced: one block has one load pipeline, an access pattern that touches 32 lines per instruction
// costs 32 of its cycles); a warp owns 8 consecutive 32-item rows of the tile.  Returns the total (to every thread).
template <class T, class Item, class Out>
__device__ __forceinline__ T block_scan_exclusive(int n, Item item, Out out) {
    constexpr int R = 8;
    __shared__ T warp_tot[32];
    __shared__ T carry_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024 * R) {
        const int i0 = base + warp * (32 * R) + lane;
        T v[R], inc[R];
#pragma unroll
        for (int j = 0; j < R; ++j) v[j] = (i0 + 32 * j < n) ? item(i0 + 32 * j) : T(0);
        T off = 0;   // sum of the warp's earlier rows
#pragma unroll
        for (int j = 0; j < R; ++j) {
            T x = v[j];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const T u = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += u;
            }
            inc[j] = off + x;
            off += __shfl_sync(0xffffffffu, x, 31);
        }
        if (lane == 0) warp_tot[warp] = off;
        __syncthreads();
        if (warp == 0) {
            T w = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const T u = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += u;
            }
            warp_tot[lane] = w;   // inclusive over warps
        }
        __syncthreads();
        const T carry = carry_s;
        const T before = carry + (warp > 0 ? warp_tot[warp - 1] : T(0));
#pragma unroll
        for (int j = 0; j < R; ++j)
            if (i0 + 32 * j < n) out(i0 + 32 * j, before + inc[j] - v[j]);
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + warp_tot[31];
        __syncthreads();
    }
    return carry_s;
}

// Both prefix sums of the cell sort in ONE launch (the per-key counts are short: bins x species): block 0 scans the
// counts in key order (bin-major) -> cstart, block 1 scans them species-major -> rstartT (first row of (species, bin)).
constexpr int kScanThreads = 1024, kScanMaxKeys = 1 << 18;
__global__ void __launch_bounds__(kScanThreads) key_scan_kernel(int nkeys, int ncell, int S, const int* __restrict__ cnt,
                                                               int* __restrict__ cstart, int* __restrict__ rstartT) {
    if (blockIdx.x == 0) {
        block_scan_exclusive<int>(
            nkeys + 1, [&](int t) { return t < nkeys ? cnt[t] : 0; }, [&](int t, int v) { cstart[t] = v; });
    } else {
        block_scan_exclusive<int>(
            nkeys + 1,
            [&](int t) {
                if (t >= nkeys) return 0;
                const int s = t / ncell, bin = t - s * ncell;   // species-major position t = s * ncell + bin
                return cnt[bin * S + s];
            },
            [&](int t, int v) { rstartT[t] = v; });
    }
}

// One warp per bin: order every (bin, species) run by original index (the atomics of bin_count_kernel hand out arbitrary
// ranks; the cell order must not depend on them) and write the cell-ordered atom records of the bin.  BATCH: the bin's
// structure gives the Geom and goes to bg.astr.
template <bool BATCH>
__global__ void sort_gather_kernel(int ncell, int64_t N, const double* __restrict__ pos, const int* __restrict__ cstart,
                                   const int* __restrict__ rstartT, Geom g_call, int S, int* __restrict__ order,
                                   AtomRec* __restrict__ atoms, int* __restrict__ abin, int* __restrict__ rowof,
                                   BatchGeom bg = BatchGeom{}) {
    const int lane = threadIdx.x & 31;
    const int bin = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (bin >= ncell) return;
    int sb = 0;
    if constexpr (BATCH) sb = batch_of(bg.bin_base, bg.B, bin);
    const Geom& g = env_geom<BATCH>(g_call, bg, sb);
    for (int s = 0; s < S; ++s) {
        const int k = bin * S + s;
        const int b = cstart[k], e = cstart[k + 1];
        if (e - b > 32) {                                  // rare: insertion sort by one lane, as long as it takes
            if (lane == 0) {
                for (int i = b + 1; i < e; ++i) {
                    const int v = order[i];
                    int j = i - 1;
                    while (j >= b && order[j] > v) {
                        order[j + 1] = order[j];
                        --j;
                    }
                    order[j + 1] = v;
                }
            }
            __syncwarp();
        } else if (e - b > 1) {
            const int len = e - b;
            const int v = lane < len ? order[b + lane] : 0x7fffffff;
            int rank = 0;
            for (int t = 0; t < len; ++t) rank += (__shfl_sync(0xffffffffu, v, t) < v) ? 1 : 0;   // indices are distinct
            __syncwarp();
            if (lane < len) order[b + rank] = v;
            __syncwarp();
        }
        const int row0 = rstartT[s * ncell + bin];
        for (int c = b + lane; c < e; c += 32) {
            const int i = order[c];
            const double x = pos[3 * (int64_t)i], y = pos[3 * (int64_t)i + 1], z = pos[3 * (int64_t)i + 2];
            int b3[3], w[3];
            frac_bin(g, x, y, z, b3, w);
            atoms[c] = atom_rec(x, y, z, i, s, w);
            abin[c] = bin;
            rowof[c] = row0 + (c - b);
            if constexpr (BATCH) bg.astr[c] = sb;
        }
    }
}

static int scan_exclusive_int(sgpr_context* h, const int* in, int* out, int n, cudaStream_t st) {
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, n, st);
    SGPR_TRY(h->scan_tmp.ensure(tmp));
    SGPR_CUDA(cub::DeviceScan::ExclusiveSum(h->scan_tmp.p, tmp, in, out, n, st));
    return SGPR_OK;
}

int scan_exclusive_ll(sgpr_context* h, const long long* in, long long* out, int n, cudaStream_t st) {
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, n, st);
    SGPR_TRY(h->scan_tmp.ensure(tmp));
    SGPR_CUDA(cub::DeviceScan::ExclusiveSum(h->scan_tmp.p, tmp, in, out, n, st));
    return SGPR_OK;
}

// Workspace layout after cell_sort (all int32 unless noted):
//   cnt     [nkeys+1]   atoms per key (last entry 0 so the exclusive scan yields the total)
//   cstart  [nkeys+1]   first cell-order index of each key
//   rstart  [2*(nkeys+1)]  transposed counts (cub path), then the species-major scan: first row of (species, bin)
//   keyrank [2N]        key per original atom, arbitrary rank within key
//   order   [N]         original index of cell-order atom c
//   atoms   [N] AtomRec ; rowof [2N]: abin[c], rowof[c]
//   errflag             error flags (single structure) and the pair cursor; bg->err (batch), bg->astr [N] (batch)
// bg: a batch (sgpr_predict_batch) -- bins of all its structures, keys structure-major (bin_count_kernel<true>); its
// errors are reported by neighbor_build's sizing step.
int cell_sort(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const Geom& g, cudaStream_t st,
              const BatchGeom* bg) {
    const int S = h->S;
    const int ncell = bg ? bg->ncell : g.ncell;
    const int nkeys = ncell * S;
    SGPR_TRY(h->cnt.ensure(sizeof(int) * (nkeys + 1)));
    SGPR_TRY(h->cstart.ensure(sizeof(int) * (nkeys + 1)));
    SGPR_TRY(h->rstart.ensure(sizeof(int) * 2 * (nkeys + 1)));
    SGPR_TRY(h->keyrank.ensure(sizeof(int) * 2 * (N + 1)));
    SGPR_TRY(h->order.ensure(sizeof(int) * (N + 1)));
    SGPR_TRY(h->atoms.ensure(sizeof(AtomRec) * (N + 1)));
    SGPR_TRY(h->rowof.ensure(sizeof(int) * 2 * (N + 1)));
    int* cnt = h->cnt.as<int>();
    int* cstart = h->cstart.as<int>();
    int* cntT = h->rstart.as<int>();
    int* rstartT = cntT + (nkeys + 1);
    int* key = h->keyrank.as<int>();
    int* rank = key + (N + 1);
    int* err = h->errflag.as<int>();
    const BatchGeom bgv = bg ? *bg : BatchGeom{};
    SGPR_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * (nkeys + 1), st));
    SGPR_CUDA(cudaMemsetAsync(err, 0, kErrflagBytes, st));   // error flags and the pair cursor
    if (bg) SGPR_CUDA(cudaMemsetAsync(bg->err, 0x7f, sizeof(unsigned long long) * 2, st));
    const int T = 256;
    const int nblkN = (int)((N + T - 1) / T);
    const int nblkK = (nkeys + T - 1) / T;
    if (N > 0)
        (bg ? bin_count_kernel<true> : bin_count_kernel<false>)<<<nblkN, T, 0, st>>>(N, pos_d, Z_d, h->ztab.as<int>(), g, S,
                                                                                     cnt, key, rank, err, bgv);
    int launches = 4;
    if (h->nl_lean && nkeys + 1 <= kScanMaxKeys) {
        // both scans in one launch (< 2^18 bin x species keys)
        key_scan_kernel<<<2, kScanThreads, 0, st>>>(nkeys, ncell, S, cnt, cstart, rstartT);
    } else {
        SGPR_CUDA(cudaMemsetAsync(cntT, 0, sizeof(int) * (nkeys + 1), st));
        transpose_cnt_kernel<<<nblkK, T, 0, st>>>(ncell, S, cnt, cntT);
        SGPR_TRY(scan_exclusive_int(h, cnt, cstart, nkeys + 1, st));
        SGPR_TRY(scan_exclusive_int(h, cntT, rstartT, nkeys + 1, st));
        launches = 8;   // transpose + 2 cub scans (2 kernels each) instead of key_scan
    }
    if (N > 0) {
        scatter_order_kernel<<<nblkN, T, 0, st>>>(N, key, rank, cstart, h->order.as<int>());
        (bg ? sort_gather_kernel<true> : sort_gather_kernel<false>)<<<(ncell + 7) / 8, 256, 0, st>>>(
            ncell, N, pos_d, cstart, rstartT, g, S, h->order.as<int>(), h->atoms.as<AtomRec>(), h->rowof.as<int>(),
            h->rowof.as<int>() + (N + 1), bgv);
    }
    h->stats.kernel_launches += launches;
    SGPR_CUDA(cudaGetLastError());
    return SGPR_OK;
}

// ---------------------------------------------------------------------------------
// neighbour search: one warp per atom, lanes over the candidates of a bin run
// ---------------------------------------------------------------------------------
// exact image shift  ((S0*c0 + S1*c1) + S2*c2)  in the reference's rounding sequence (no FMA)
__device__ __forceinline__ void shift_vec(const Geom& g, int S0, int S1, int S2, double& s0, double& s1, double& s2) {
    const double a = (double)S0, b = (double)S1, c = (double)S2;
    s0 = __dadd_rn(__dadd_rn(__dmul_rn(a, g.cell[0]), __dmul_rn(b, g.cell[3])), __dmul_rn(c, g.cell[6]));
    s1 = __dadd_rn(__dadd_rn(__dmul_rn(a, g.cell[1]), __dmul_rn(b, g.cell[4])), __dmul_rn(c, g.cell[7]));
    s2 = __dadd_rn(__dadd_rn(__dmul_rn(a, g.cell[2]), __dmul_rn(b, g.cell[5])), __dmul_rn(c, g.cell[8]));
}

// Accept/reject exactly as the reference:  sqrt(sum(r*r)) < rc  with  r = (x_j - x_i) + shift.
// (sh0,sh1,sh2) is the shift of the bin run, valid when i and j carry the same wrap shift (the
// common case); the square root is only evaluated when d^2 is within 1e-14 of rc^2, elsewhere
// comparing squares gives the same answer.
__device__ __forceinline__ bool pair_test(const Geom& g, const AtomRec& ai, const AtomRec& aj, int sx, int sy, int sz,
                                          double sh0, double sh1, double sh2, double rc2_lo, double rc2_hi, bool same) {
    bool zero_shift = (sx | sy | sz) == 0;
    if ((unsigned)(aj.meta >> 40) != (unsigned)(ai.meta >> 40)) {
        // image shift relative to the positions as given:  S = S_bin - w_j + w_i
        const int S0 = sx - meta_w(aj.meta, 0) + meta_w(ai.meta, 0);
        const int S1 = sy - meta_w(aj.meta, 1) + meta_w(ai.meta, 1);
        const int S2 = sz - meta_w(aj.meta, 2) + meta_w(ai.meta, 2);
        zero_shift = (S0 | S1 | S2) == 0;
        shift_vec(g, S0, S1, S2, sh0, sh1, sh2);
    }
    if (same && zero_shift) return false;
    const double rx = __dadd_rn(__dadd_rn(aj.x, -ai.x), sh0);
    const double ry = __dadd_rn(__dadd_rn(aj.y, -ai.y), sh1);
    const double rz = __dadd_rn(__dadd_rn(aj.z, -ai.z), sh2);
    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(rx, rx), __dmul_rn(ry, ry)), __dmul_rn(rz, rz));
    bool acc = d2 < rc2_lo;
    if (!acc && d2 <= rc2_hi) acc = __dsqrt_rn(d2) < g.rc;
    return acc;
}

// bin index n + periodic wrap -> (wrapped bin, image shift); false if outside a non-periodic box
__device__ __forceinline__ bool wrap_bin(int n, int nb, int pbc, int& nw, int& sh) {
    sh = 0;
    nw = n;
    if (pbc) {
        while (nw < 0) {
            nw += nb;
            --sh;
        }
        while (nw >= nb) {
            nw -= nb;
            ++sh;
        }
        return true;
    }
    return n >= 0 && n < nb;
}

constexpr int kMaskSlots = 64;

// One warp per environment.  COUNT pass: distance tests, per-species counts (packed 16-bit
// per-lane counters, one warp reduction at the end), accept masks per candidate batch and halo
// marks.  FILL pass: replays the traversal, takes the accept bits from the masks and writes the
// pairs species-sorted (per-species ballots give each accepted candidate its rank).
// BATCH: a batch of structures (sgpr_predict_batch) -- each environment reads its structure's Geom, and its stencil
// stays inside that structure's bins (bg.bin_base); same traversal, pair_test and pair order as a call on the structure
template <bool FILL, int NS, bool BATCH = false>
__global__ void __launch_bounds__(256) neighbor_kernel(int env0, int n_env, const int* __restrict__ active,
                                                       const AtomRec* __restrict__ atoms, const int* __restrict__ abin,
                                                       const int* __restrict__ cstart, Geom g_call, int S,
                                                       int* __restrict__ nl_cnt, const long long* __restrict__ nl_first,
                                                       const long long* __restrict__ cursor, long long cap,
                                                       longlong2* __restrict__ rows, PairRec* __restrict__ pairs,
                                                       unsigned char* __restrict__ mark, unsigned* __restrict__ masks,
                                                       BatchGeom bg = BatchGeom{}) {
    const int lane = threadIdx.x & 31;
    int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (wid >= n_env) return;
    const int k_env = wid;   // index among this launch's environments (nl_first)
    wid += env0;  // index into the active list / the neighbour-list rows
    const int c = active ? active[wid] : wid;
    int sb = 0, bbase = 0;
    if constexpr (BATCH) {
        sb = bg.astr[c];
        bbase = bg.bin_base[sb];
    }
    const Geom& g = env_geom<BATCH>(g_call, bg, sb);
    const AtomRec ai = atoms[c];
    int bin = abin[c] - bbase;
    const int bz = bin % g.nb[2];
    bin /= g.nb[2];
    const int by = bin % g.nb[1];
    const int bx = bin / g.nb[1];
    int count[NS];
    long long base[NS];
    unsigned long long pc0 = 0ull, pc1 = 0ull;   // COUNT: packed per-lane counters, 16 bits per species
    int slot = 0;
    unsigned* my_masks = masks + (size_t)wid * kMaskSlots;
    const double rc2 = g.rc * g.rc;
    const double rc2_lo = rc2 * (1.0 - 1e-14), rc2_hi = rc2 * (1.0 + 1e-14);
#pragma unroll
    for (int s = 0; s < NS; ++s) count[s] = 0;
    bool fits = true;
    if (FILL) {
        // this launch's rows follow the pairs already reserved on the cursor (block-per-bin rows of the same step)
        const long long row0 = *cursor + nl_first[k_env];
        long long o = row0;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            base[s] = o;
            if (s < S) o += nl_cnt[(long long)wid * S + s];
        }
        if (lane == 0) rows[wid] = make_longlong2(row0, o);
        fits = o <= cap;   // an invalid warm step writes no pairs (nl_finish_kernel empties its rows)
    }
    for (int dx = -g.reach[0]; dx <= g.reach[0]; ++dx) {
        int nx, sx;
        if (!wrap_bin(bx + dx, g.nb[0], g.pbc[0], nx, sx)) continue;
        for (int dy = -g.reach[1]; dy <= g.reach[1]; ++dy) {
            int ny, sy;
            if (!wrap_bin(by + dy, g.nb[1], g.pbc[1], ny, sy)) continue;
            // z bins of this (x,y) column: contiguous in cell order -> one merged run when the
            // stencil does not wrap (or leave the box) inside the column
            const int zlo = bz - g.reach[2], zhi = bz + g.reach[2];
            const bool merged = (zlo >= 0 && zhi < g.nb[2]);
            for (int dz = merged ? 0 : -g.reach[2]; dz <= (merged ? 0 : g.reach[2]); ++dz) {
                int nz, sz = 0, nz_last;
                if (merged) {
                    nz = zlo;
                    nz_last = zhi;
                } else {
                    if (!wrap_bin(bz + dz, g.nb[2], g.pbc[2], nz, sz)) continue;
                    nz_last = nz;
                }
                const int b2 = bbase + (nx * g.nb[1] + ny) * g.nb[2] + nz;
                const int b3 = bbase + (nx * g.nb[1] + ny) * g.nb[2] + nz_last;
                const int beg = cstart[b2 * S], end = cstart[b3 * S + S];
                double sh0 = 0.0, sh1 = 0.0, sh2 = 0.0;
                if (!FILL) shift_vec(g, sx, sy, sz, sh0, sh1, sh2);
                for (int p0 = beg; p0 < end; p0 += 32) {
                    const int p = p0 + lane;
                    bool acc = false;
                    int sp = 0;
                    if (FILL && slot < kMaskSlots) {
                        acc = (my_masks[slot] >> lane) & 1u;
                        if (acc) sp = meta_species(atoms[p].meta);
                    } else if (p < end) {
                        const AtomRec aj = atoms[p];
                        sp = meta_species(aj.meta);
                        if (FILL) shift_vec(g, sx, sy, sz, sh0, sh1, sh2);   // rare: more than kMaskSlots batches
                        acc = pair_test(g, ai, aj, sx, sy, sz, sh0, sh1, sh2, rc2_lo, rc2_hi, p == c);
                    }
                    if (!FILL) {
                        if (acc) {
                            if (mark) mark[p] = 1;   // atoms whose environment the owner needs (halo)
                            const unsigned long long one = 1ull << (16 * (sp & 3));
                            if (NS <= 4 || sp < 4) pc0 += one;
                            else pc1 += one;
                        }
                        if (slot < kMaskSlots) {
                            const unsigned m_all = __ballot_sync(0xffffffffu, acc);
                            if (lane == 0) my_masks[slot] = m_all;
                        }
                    } else {
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            const unsigned m = __ballot_sync(0xffffffffu, acc && sp == s);
                            if (fits && acc && sp == s) {
                                PairRec pr;
                                pr.j = p;
                                pr.sb[0] = (signed char)sx;
                                pr.sb[1] = (signed char)sy;
                                pr.sb[2] = (signed char)sz;
                                pr.sp = (unsigned char)sp;
                                pairs[base[s] + count[s] + __popc(m & ((1u << lane) - 1u))] = pr;
                            }
                            count[s] += __popc(m);
                        }
                    }
                    ++slot;
                }
            }
        }
    }
    if (!FILL) {
        // warp sums of the packed counters (each species total < 65536)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            pc0 += __shfl_xor_sync(0xffffffffu, pc0, o);
            if (NS > 4) pc1 += __shfl_xor_sync(0xffffffffu, pc1, o);
        }
        if (lane == 0) {
#pragma unroll
            for (int s = 0; s < NS; ++s)
                if (s < S) nl_cnt[(long long)wid * S + s] = (int)(((s < 4 ? pc0 : pc1) >> (16 * (s & 3))) & 0xffffull);
        }
    }
}

// ---------------------------------------------------------------------------------
// neighbour search, one BLOCK per bin (the path for all but tiny systems), in ONE pass: every atom of a bin walks the
// same stencil, so the block gathers the candidates of the stencil once into shared memory -- already shifted to the
// right periodic image -- and its warps test their atoms against that tile without touching global memory.  The
// accept bits stay in shared memory; the block then reserves the rows of its atoms in nl_pairs with one atomicAdd on
// the pair cursor and writes the pairs from the bits.  Inside a row the pairs are ordered by species, then tile, then
// lane, then slot (the descriptor kernels sum a row in this order); the accept rule is neighbor_kernel's: the
// shared-memory test decides everything except d^2 within 1e-11 of rc^2, which goes through pair_test (the reference's
// rounding sequence).
// Rows land in nl_pairs in whatever order the atomics hand out the segments: consumers read [begin, end) of a row.
// ---------------------------------------------------------------------------------
constexpr int kBinThreads = 256, kBinCap = 1024, kRunChunk = 128;
constexpr int kBinAtoms = 32;   // atoms per round of a block (one lane each in the reservation); crowded bins take several

template <int NS>
__global__ void __launch_bounds__(kBinThreads, 4) neighbor_bin_kernel(int c_begin, int c_end, int env0,
                                                                   const AtomRec* __restrict__ atoms,
                                                                   const int* __restrict__ cstart,
                                                                   const __grid_constant__ Geom g, int S,
                                                                   long long* __restrict__ cursor, long long cap,
                                                                   longlong2* __restrict__ rows, PairRec* __restrict__ pairs,
                                                                   unsigned char* __restrict__ mark) {
    // candidate image relative to the bin's first atom, in float (x, y, z), and w = |x| + |y| + |z| of the unshifted and
    // shifted absolute coordinates (rounding bound of the double-precision test)
    __shared__ float4 rel[kBinCap];
    __shared__ unsigned maxabs_u;            // running max of the relative coordinates' 1-norm (float bits)
    __shared__ int pj[kBinCap];
    __shared__ unsigned code[kBinCap];       // bin shift (3 x int8) | species << 24
    __shared__ int run_beg[kRunChunk], run_pre[kRunChunk + 1];
    __shared__ unsigned run_sh[kRunChunk];
    __shared__ unsigned long long acc_s[kBinAtoms][32];   // accept bits of an atom: bit k of lane l = candidate (slot k, l)
    __shared__ int cnt_s[kBinAtoms][NS];     // accepted candidates per species over the whole stencil
    __shared__ int done_s[kBinAtoms][NS];    // pairs per species written by earlier tiles
    __shared__ long long row_s[kBinAtoms];   // first pair of the row
    __shared__ int fits_s;                   // the round's segment lies inside nl_pairs
    __shared__ unsigned smask_s[NS][32];     // bit b of [s][l]: candidate (batch b, lane l) of the tile has species s
    const int bin = blockIdx.x;
    const int lo = max(cstart[bin * S], c_begin), hi = min(cstart[(bin + 1) * S], c_end);
    if (lo >= hi) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NW = kBinThreads / 32;
    if (threadIdx.x == 0) maxabs_u = 0u;
    double refx, refy, refz;   // the bin's first atom, wrapped into the box: origin of the float coordinates
    {
        const AtomRec a0 = atoms[lo];
        double w0, w1, w2;
        shift_vec(g, meta_w(a0.meta, 0), meta_w(a0.meta, 1), meta_w(a0.meta, 2), w0, w1, w2);
        refx = a0.x - w0;
        refy = a0.y - w1;
        refz = a0.z - w2;
    }
    const int bz = bin % g.nb[2], by = (bin / g.nb[2]) % g.nb[1], bx = bin / (g.nb[2] * g.nb[1]);
    const int zlo = bz - g.reach[2], zhi = bz + g.reach[2];
    const bool merged = (zlo >= 0 && zhi < g.nb[2]);   // z stencil contiguous in cell order: one run per column
    const int nyr = 2 * g.reach[1] + 1, nzr = merged ? 1 : 2 * g.reach[2] + 1;
    const int nruns = (2 * g.reach[0] + 1) * nyr * nzr;
    const double rc2 = g.rc * g.rc;
    const double fast_lo = rc2 * (1.0 - 1e-11), fast_hi = rc2 * (1.0 + 1e-11);
    const double rc2_lo = rc2 * (1.0 - 1e-14), rc2_hi = rc2 * (1.0 + 1e-14);

    // runs r0 .. r0+nr-1 of the stencil: first candidate, count (run_pre: exclusive prefix) and bin shift
    auto stage_runs = [&](int r0, int nr) {
        __syncthreads();   // the previous tile is still being read
        for (int t = threadIdx.x; t < NS * 32; t += kBinThreads) smask_s[t >> 5][t & 31] = 0u;
        for (int t = threadIdx.x; t < nr; t += kBinThreads) {
            const int r = r0 + t;
            const int iz = r % nzr, iy = (r / nzr) % nyr, ix = r / (nzr * nyr);
            int nx, sx, ny, sy, nz = zlo, sz = 0, nz_last = zhi;
            bool ok = wrap_bin(bx + ix - g.reach[0], g.nb[0], g.pbc[0], nx, sx) &&
                      wrap_bin(by + iy - g.reach[1], g.nb[1], g.pbc[1], ny, sy);
            if (ok && !merged) {
                ok = wrap_bin(bz + iz - g.reach[2], g.nb[2], g.pbc[2], nz, sz);
                nz_last = nz;
            }
            int beg = 0, len = 0;
            if (ok) {
                const int col = (nx * g.nb[1] + ny) * g.nb[2];
                beg = cstart[(col + nz) * S];
                len = cstart[(col + nz_last) * S + S] - beg;
            }
            run_beg[t] = beg;
            run_pre[t + 1] = len;
            run_sh[t] = (unsigned)(sx & 0xff) | ((unsigned)(sy & 0xff) << 8) | ((unsigned)(sz & 0xff) << 16);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            run_pre[0] = 0;
            for (int t = 0; t < nr; ++t) run_pre[t + 1] += run_pre[t];
        }
        __syncthreads();
    };
    // candidates t0 .. t0+n-1 of the staged runs into the tile
    auto stage_tile = [&](int nr, int t0, int n) {
        if (t0 > 0) {
            __syncthreads();   // the previous tile is still being read
            for (int t = threadIdx.x; t < NS * 32; t += kBinThreads) smask_s[t >> 5][t & 31] = 0u;
            __syncthreads();
        }
        float my_max = 0.0f;
        for (int q = threadIdx.x; q < n; q += kBinThreads) {
            const int gq = t0 + q;
            int a = 0, b = nr;          // last run with run_pre[a] <= gq
            while (b - a > 1) {
                const int mid = (a + b) >> 1;
                if (run_pre[mid] <= gq) a = mid;
                else b = mid;
            }
            const int p = run_beg[a] + (gq - run_pre[a]);
            const AtomRec aj = atoms[p];
            const unsigned sh = run_sh[a];
            double s0, s1, s2;
            shift_vec(g, (int)(signed char)(sh & 0xff) - meta_w(aj.meta, 0), (int)(signed char)((sh >> 8) & 0xff) - meta_w(aj.meta, 1),
                      (int)(signed char)((sh >> 16) & 0xff) - meta_w(aj.meta, 2), s0, s1, s2);
            const float fx = (float)((aj.x + s0) - refx), fy = (float)((aj.y + s1) - refy), fz = (float)((aj.z + s2) - refz);
            rel[q] = make_float4(fx, fy, fz,
                                 (float)(fabs(aj.x) + fabs(aj.y) + fabs(aj.z) + fabs(s0) + fabs(s1) + fabs(s2)) * 1.0001f);
            my_max = fmaxf(my_max, fabsf(fx) + fabsf(fy) + fabsf(fz));
            pj[q] = p;
            code[q] = sh | ((unsigned)meta_species(aj.meta) << 24);
            atomicOr(&smask_s[meta_species(aj.meta)][q & 31], 1u << (q >> 5));
        }
        {
            const unsigned m = __reduce_max_sync(0xffffffffu, __float_as_uint(my_max));   // floats >= 0 order as uints
            if (lane == 0 && m > 0u) atomicMax(&maxabs_u, m);
        }
        __syncthreads();
    };
    // one atom against the tile: COUNT pass (accept bits, per-species counts, halo marks) or EMIT pass (pairs)
    auto visit = [&](bool emit, int c, int a, int n, int slot_base) {
        const AtomRec ai = atoms[c];
        const float maxabs = __uint_as_float(maxabs_u);
        double w0, w1, w2;
        shift_vec(g, meta_w(ai.meta, 0), meta_w(ai.meta, 1), meta_w(ai.meta, 2), w0, w1, w2);
        const double xi = ai.x - w0, yi = ai.y - w1, zi = ai.z - w2;   // the atom's image inside the box
        // |d2 - d2_reference| <= ~2 rc sqrt(3) * (rounding of the coordinates involved): the band in which the
        // shared-memory test may disagree with the reference's rounding sequence grows with the coordinates'
        // magnitude (unwrapped trajectories far from the origin)
        const double imag = fabs(ai.x) + fabs(ai.y) + fabs(ai.z) + fabs(w0) + fabs(w1) + fabs(w2);
        // distance test of candidate q.  Float coordinates relative to the bin decide everything farther from the
        // cutoff sphere than their rounding error: with coordinates of 1-norm <= m the float d2 is off by less
        // than 2^-24 (7 m |d| + 5 d^2) <= 2^-19 (m^2 + rc^2) wherever a decision is taken -- the margin is 4x
        // that.  Inside the margin (and for d2 ~ 0: the atom itself) the double-precision test decides, with the
        // reference's exact rounding sequence only in its own, much narrower band.
        const float fxi = (float)(xi - refx), fyi = (float)(yi - refy), fzi = (float)(zi - refz);
        const float mx = fmaxf(maxabs, fabsf(fxi) + fabsf(fyi) + fabsf(fzi));
        const float margin = 7.62939453125e-6f * (mx * mx + (float)rc2);   // 2^-17
        const float lo_f = (float)rc2 - margin, hi_f = (float)rc2 + margin;
        // candidates the float test leaves undecided (rare)
        auto exact = [&](int q) -> bool {
            const float4 cq = rel[q];
            const unsigned cd = code[q];
            const int p = pj[q];
            if (p == c && (cd & 0xffffffu) == 0u) return false;   // the atom itself (zero image shift)
            const AtomRec aj = atoms[p];
            const int sx = (int)(signed char)(cd & 0xff), sy = (int)(signed char)((cd >> 8) & 0xff),
                      sz = (int)(signed char)((cd >> 16) & 0xff);
            double s0, s1, s2;
            shift_vec(g, sx - meta_w(aj.meta, 0), sy - meta_w(aj.meta, 1), sz - meta_w(aj.meta, 2), s0, s1, s2);
            const double dx = (aj.x + s0) - xi, dy = (aj.y + s1) - yi, dz = (aj.z + s2) - zi;
            const double d2 = dx * dx + dy * dy + dz * dz;
            const double band = 3.6e-15 * g.rc * ((double)cq.w + imag);   // 2^-48 rc (|x_j| + |x_i| + shifts)
            if (d2 < fast_lo - band) return true;
            if (d2 > fast_hi + band) return false;
            double sh0, sh1, sh2;
            shift_vec(g, sx, sy, sz, sh0, sh1, sh2);
            return pair_test(g, ai, aj, sx, sy, sz, sh0, sh1, sh2, rc2_lo, rc2_hi, false);
        };
        auto test = [&](int q) -> bool {
            const float4 cq = rel[q];
            const float ex = cq.x - fxi, ey = cq.y - fyi, ez = cq.z - fzi;
            const float d2f = fmaf(ex, ex, fmaf(ey, ey, ez * ez));
            if (d2f > hi_f) return false;
            if (d2f < lo_f && d2f > margin) return true;
            return exact(q);
        };
        // per-lane counts of the accepted candidates in w by species, packed 16 bits per species
        auto species_counts = [&](unsigned w, unsigned long long& pc0, unsigned long long& pc1) {
            pc0 = pc1 = 0ull;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const unsigned long long v = (unsigned long long)__popc(w & smask_s[s][lane]) << (16 * (s & 3));
                if (s < 4) pc0 += v;
                else pc1 += v;
            }
        };
        // accept bits of an atom: one 64-bit word per lane, bit k = candidate (slot k, this lane); slots beyond the
        // word (more than 2048 candidates) are tested again by the EMIT pass
        const int nb_tile = (n + 31) >> 5;
        const int nb_masked = max(0, min(nb_tile, 64 - slot_base));   // batches of this tile covered by the word
        if (!emit) {
            // the float test over the tile (a tile has at most 32 batches: one bit each), undecided candidates after it
            unsigned w = 0u, undecided = 0u;
            for (int b = 0; b < nb_tile; ++b) {
                const int q = b * 32 + lane;
                if (q < n) {
                    const float4 cq = rel[q];
                    const float ex = cq.x - fxi, ey = cq.y - fyi, ez = cq.z - fzi;
                    const float d2f = fmaf(ex, ex, fmaf(ey, ey, ez * ez));
                    if (d2f <= hi_f) {
                        if (d2f < lo_f && d2f > margin) w |= 1u << b;
                        else undecided |= 1u << b;
                    }
                }
            }
            for (unsigned t = undecided; t; t &= t - 1) {
                const int b = __ffs(t) - 1;
                if (exact(b * 32 + lane)) w |= 1u << b;
            }
            if (mark)   // atoms whose environment the owner needs (halo)
                for (unsigned t = w; t; t &= t - 1) mark[pj[(__ffs(t) - 1) * 32 + lane]] = 1;
            if (nb_masked > 0) acc_s[a][lane] = (slot_base > 0 ? acc_s[a][lane] : 0ull) | ((unsigned long long)w << slot_base);
            unsigned long long pc0, pc1;
            species_counts(w, pc0, pc1);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                pc0 += __shfl_xor_sync(0xffffffffu, pc0, o);
                if (NS > 4) pc1 += __shfl_xor_sync(0xffffffffu, pc1, o);
            }
            if (lane == 0) {
#pragma unroll
                for (int s = 0; s < NS; ++s) cnt_s[a][s] += (int)(((s < 4 ? pc0 : pc1) >> (16 * (s & 3))) & 0xffffull);
            }
            return;
        }
        // pairs of one species are contiguous; inside a species: tile, then lane, then slot
        long long start[NS];
        {
            long long o = row_s[a];
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                start[s] = o + done_s[a][s];
                o += cnt_s[a][s];
            }
        }
        auto emit_pair = [&](int q, unsigned long long& run0, unsigned long long& run1) {
            const unsigned cd = code[q];
            const int sp = (int)(cd >> 24);
            long long b = 0;
#pragma unroll
            for (int s = 0; s < NS; ++s)
                if (sp == s) b = start[s];
            unsigned long long& run = (NS <= 4 || sp < 4) ? run0 : run1;
            const int r = (int)((run >> (16 * (sp & 3))) & 0xffffull);
            run += 1ull << (16 * (sp & 3));
            PairRec pr;
            pr.j = pj[q];
            pr.sb[0] = (signed char)(cd & 0xff);
            pr.sb[1] = (signed char)((cd >> 8) & 0xff);
            pr.sb[2] = (signed char)((cd >> 16) & 0xff);
            pr.sp = (unsigned char)sp;
            pairs[b + r] = pr;
        };
        // this lane's accepted candidates of the tile: stored bits, tested again beyond the word's reach (rare)
        unsigned w = nb_masked > 0 ? (unsigned)(acc_s[a][lane] >> slot_base) : 0u;
        if (nb_tile < 32) w &= (1u << nb_tile) - 1u;   // drop the next tile's bits
        for (int b = nb_masked; b < nb_tile; ++b) {
            const int q = b * 32 + lane;
            if (q < n && test(q)) w |= 1u << b;
        }
        unsigned long long pc0, pc1;
        species_counts(w, pc0, pc1);
        // exclusive prefix over lanes (16-bit fields cannot carry: totals < 65536)
        unsigned long long in0 = pc0, in1 = pc1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u0 = __shfl_up_sync(0xffffffffu, in0, o);
            const unsigned long long u1 = NS > 4 ? __shfl_up_sync(0xffffffffu, in1, o) : 0ull;
            if (lane >= o) {
                in0 += u0;
                in1 += u1;
            }
        }
        unsigned long long run0 = in0 - pc0, run1 = in1 - pc1;
        const unsigned long long tot0 = __shfl_sync(0xffffffffu, in0, 31);
        const unsigned long long tot1 = NS > 4 ? __shfl_sync(0xffffffffu, in1, 31) : 0ull;
        for (unsigned t = w; t; t &= t - 1) emit_pair((__ffs(t) - 1) * 32 + lane, run0, run1);
        if (lane == 0) {
#pragma unroll
            for (int s = 0; s < NS; ++s) done_s[a][s] += (int)(((s < 4 ? tot0 : tot1) >> (16 * (s & 3))) & 0xffffull);
        }
    };
    // A bin whose stencil is one tile (the common case) stages it once; otherwise both passes stage every tile.
    bool resident = false;
    auto walk = [&](bool emit, int a0, int a1) {
        int slot_base = 0;
        for (int r0 = 0; r0 < nruns; r0 += kRunChunk) {
            const int nr = min(kRunChunk, nruns - r0);
            if (!resident) stage_runs(r0, nr);
            const int total = run_pre[nr];
            for (int t0 = 0; t0 < total; t0 += kBinCap) {
                const int n = min(kBinCap, total - t0);
                if (!resident) stage_tile(nr, t0, n);
                for (int c = a0 + warp; c < a1; c += NW) visit(emit, c, c - a0, n, slot_base);
                slot_base += (n + 31) >> 5;
            }
            resident = nruns <= kRunChunk && total <= kBinCap;
        }
    };
    for (int a0 = lo; a0 < hi; a0 += kBinAtoms) {
        const int a1 = min(hi, a0 + kBinAtoms);
        if (a0 > lo) __syncthreads();   // the previous round still reads cnt_s / done_s
        for (int t = threadIdx.x; t < kBinAtoms * NS; t += kBinThreads) {
            cnt_s[t / NS][t % NS] = 0;
            done_s[t / NS][t % NS] = 0;
        }
        __syncthreads();
        walk(false, a0, a1);
        __syncthreads();
        // reserve the round's rows: one atomic per round, rows in cell order inside the segment
        if (warp == 0) {
            int tot = 0;
            if (lane < a1 - a0)
                for (int s = 0; s < S; ++s) tot += cnt_s[lane][s];
            int inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += u;
            }
            unsigned long long base = 0ull;
            if (lane == 31) base = atomicAdd(reinterpret_cast<unsigned long long*>(cursor), (unsigned long long)inc);
            base = __shfl_sync(0xffffffffu, base, 31);
            const long long b0 = (long long)base + (inc - tot);
            if (lane < a1 - a0) {
                row_s[lane] = b0;
                rows[a0 + lane - c_begin + env0] = make_longlong2(b0, b0 + tot);
            }
            if (lane == 31) fits_s = (long long)base + inc <= cap ? 1 : 0;   // else: count only (the sizing step re-runs)
        }
        __syncthreads();
        if (fits_s) walk(true, a0, a1);
    }
}

static void launch_neighbor_bins(sgpr_context* h, const Geom& g, int c_begin, int c_end, int env0, unsigned char* mark,
                                 cudaStream_t st) {
    const int nblk = g.ncell, T = kBinThreads, S = h->S;
    const AtomRec* atoms = h->atoms.as<AtomRec>();
    const int* cstart = h->cstart.as<int>();
    long long* cursor = pair_cursor(h);
    longlong2* rows = h->nl_rows.as<longlong2>();
    PairRec* pairs = h->nl_pairs.as<PairRec>();
    const long long cap = h->pairs_cap;
    if (S <= 1)
        neighbor_bin_kernel<1><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, cursor, cap, rows, pairs, mark);
    else if (S <= 2)
        neighbor_bin_kernel<2><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, cursor, cap, rows, pairs, mark);
    else if (S <= 4)
        neighbor_bin_kernel<4><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, cursor, cap, rows, pairs, mark);
    else
        neighbor_bin_kernel<8><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, cursor, cap, rows, pairs, mark);
    h->stats.kernel_launches += 1;
}

// the block-per-bin kernels need enough bins to fill the machine; tiny systems keep one warp per environment
static bool use_bin_kernels(const sgpr_context* h, const Geom& g) { return h->nl_mode == 2 || (g.ncell >= 64 && h->nl_mode != 1); }

// one warp per environment, environments env0 .. env0+n_env-1 (FILL: nl_first = exclusive scan of their row lengths)
template <bool FILL>
static void launch_neighbor(sgpr_context* h, cudaStream_t st, int env0, int n_env, const Geom& g, const long long* nl_first,
                            unsigned char* mark, const BatchGeom* bg) {
    const int T = 256, S = h->S;
    const int nblk = (int)(((int64_t)n_env * 32 + T - 1) / T);
    const int* active = h->active_all ? nullptr : h->active_list.as<int>();
    auto go = [&](auto kernel) {
        kernel<<<nblk, T, 0, st>>>(env0, n_env, active, h->atoms.as<AtomRec>(), h->rowof.as<int>(), h->cstart.as<int>(), g, S,
                                   h->nl_cnt.as<int>(), nl_first, pair_cursor(h), h->pairs_cap, h->nl_rows.as<longlong2>(),
                                   h->nl_pairs.as<PairRec>(), mark, h->nl_masks.as<unsigned>(), bg ? *bg : BatchGeom{});
    };
    if (bg) {
        if (S <= 1) go(neighbor_kernel<FILL, 1, true>);
        else if (S <= 2) go(neighbor_kernel<FILL, 2, true>);
        else if (S <= 4) go(neighbor_kernel<FILL, 4, true>);
        else go(neighbor_kernel<FILL, 8, true>);
    } else {
        if (S <= 1) go(neighbor_kernel<FILL, 1>);
        else if (S <= 2) go(neighbor_kernel<FILL, 2>);
        else if (S <= 4) go(neighbor_kernel<FILL, 4>);
        else go(neighbor_kernel<FILL, 8>);
    }
    h->stats.kernel_launches += 1;
}

// contig_c0 >= 0: environments env0 .. env0+n_env-1 are the atoms contig_c0 .. of the cell order -- the block-per-bin
// kernel writes their rows and pairs in one pass.  Otherwise the warp kernel counts them and nl_finish fills their rows.
static void launch_count(sgpr_context* h, int env0, int n_env, const Geom& g, unsigned char* mark, cudaStream_t st,
                         int contig_c0, const BatchGeom* bg = nullptr) {
    if (n_env <= 0) return;
    if (contig_c0 >= 0 && !bg && use_bin_kernels(h, g))
        launch_neighbor_bins(h, g, contig_c0, contig_c0 + n_env, env0, mark, st);
    else
        launch_neighbor<false>(h, st, env0, n_env, g, nullptr, mark, bg);
}

static int check_err_flags(const int* err) {
    if (err[0] == 1) {
        set_error("atomic number %d is not in the handle's species table", err[1]);
        return SGPR_ERR_SPECIES;
    }
    if (err[0] == 2) {
        set_error("an atom lies more than 120 cells outside the unit cell; wrap positions first");
        return SGPR_ERR_GEOMETRY;
    }
    return SGPR_OK;
}

// batch errors name the first structure that failed (bin_count_kernel<true>)
static int check_batch_err(const unsigned long long* berr) {
    const unsigned long long none = 0x7f7f7f7f7f7f7f7full;
    if (berr[0] != none) {
        set_error("structure %d: atomic number %d is not in the handle's species table", (int)(berr[0] >> 32),
                  (int)(unsigned)(berr[0] & 0xffffffffull));
        return SGPR_ERR_SPECIES;
    }
    if (berr[1] != none) {
        set_error("structure %d: an atom lies more than 120 cells outside the unit cell; wrap positions first", (int)berr[1]);
        return SGPR_ERR_GEOMETRY;
    }
    return SGPR_OK;
}

__global__ void row_total_kernel(int n, int S, const int* __restrict__ nl_cnt, long long* __restrict__ tot) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    long long t = 0;
    if (i < n)
        for (int s = 0; s < S; ++s) t += nl_cnt[(long long)i * S + s];
    tot[i] = t;
}

// Lean form of row totals -> exclusive scan for the rows of the warp kernel: one block walks the rows in coalesced tiles
// of 1024 with a running carry.  (A few microseconds for 1e5 rows, and one graph node instead of three: what matters for
// small systems and for the halo rows of a sharded one.)
constexpr int kRowsScanMax = 1 << 16;   // beyond: row_total + cub scan (one SM would be the bottleneck)
__global__ void __launch_bounds__(1024) rows_scan_kernel(int n, int S, const int* __restrict__ nl_cnt,
                                                         long long* __restrict__ first) {
    block_scan_exclusive<long long>(
        n + 1,
        [&](int i) -> long long {
            if (i >= n) return 0;
            if (S == 4) {
                const int4 c = *reinterpret_cast<const int4*>(nl_cnt + 4 * (long long)i);
                return (long long)c.x + c.y + c.z + c.w;
            }
            long long t = 0;
            for (int s = 0; s < S; ++s) t += nl_cnt[(long long)i * S + s];
            return t;
        },
        [&](int i, long long v) { first[i] = v; });
}

// Last node of the neighbour stage: the species row ranges go to their canonical device location (read by the GEMM set-up
// kernel and row_energy_kernel) and, on sync-free steps, the pair total and the error flags to the status block.  The
// total is the pair cursor (block-per-bin rows) plus the rows of the warp kernel.  A step is valid when the pair list fits
// the capacity sized by an earlier step and no error flag is set; an invalid step gets EMPTY rows, so that every later
// kernel stays inside its buffers -- its results are then meaningless and the sticky counter status[1] says so
// (sgpr_check / the host entry point re-run it).
__global__ void __launch_bounds__(1024) nl_finish_kernel(int na, int S, const int* __restrict__ row_first_src, int pitch_ints,
                                                         int* __restrict__ row_first_d, int do_status,
                                                         const long long* __restrict__ cursor,
                                                         const long long* __restrict__ warp_total, long long cap,
                                                         const int* __restrict__ err, long long* __restrict__ status,
                                                         longlong2* __restrict__ rows) {
    __shared__ int bad_s;
    if ((int)threadIdx.x <= S) row_first_d[threadIdx.x] = row_first_src[(size_t)threadIdx.x * pitch_ints];
    if (!do_status) return;
    if (threadIdx.x == 0) {
        const long long total = *cursor + (warp_total ? *warp_total : 0);
        const bool bad = total > cap || err[0] != 0;
        status[0] = total;
        status[6] = bad ? 1 : 0;
        if (bad) {
            status[1] += 1;
            status[2] = err[0];
            status[3] = err[1];
            status[4] = total;
            status[5] = cap;
        }
        bad_s = bad ? 1 : 0;
    }
    __syncthreads();
    if (bad_s)
        for (int i = threadIdx.x; i < na; i += blockDim.x) rows[i] = make_longlong2(0, 0);
}

// Rows of the environments the block-per-bin kernel has not written (it writes the first n_contig, a contiguous range of
// the cell order from contig_c0, when use_bin_kernels): per-environment counts of the warp kernel -> exclusive scan ->
// fill behind the cursor.  A sizing step (warm = false) then synchronises for the pair total, the error flags and the
// species row ranges; when the list does not fit it grows the capacity with head room (the following steps of a
// trajectory reuse it without asking the device) and runs the block-per-bin kernel again, whose pairs did not fit.
static int nl_finish(sgpr_context* h, const Geom& g, cudaStream_t st, const int* row_first_src, int row_first_pitch,
                     int64_t* n_pairs, int contig_c0, int n_contig, bool warm, const BatchGeom* bg = nullptr) {
    const int S = h->S;
    const int na = (int)h->n_active;
    const int done = (n_contig > 0 && !bg && use_bin_kernels(h, g)) ? n_contig : 0;
    const int nw = na - done;
    SGPR_TRY(h->nl_first.ensure(sizeof(long long) * 2 * ((size_t)nw + 1)));
    SGPR_TRY(h->row_first_d.ensure(sizeof(int) * (SGPR_MAX_SPECIES + 2)));
    SGPR_TRY(h->status_d.ensure(sizeof(long long) * 8));
    long long* first = h->nl_first.as<long long>();
    long long* cursor = pair_cursor(h);
    const int T = 256;
    if (nw > 0) {
        const int* cnt = h->nl_cnt.as<int>() + (size_t)done * S;
        if (h->nl_lean && nw + 1 <= kRowsScanMax) {
            rows_scan_kernel<<<1, 1024, 0, st>>>(nw, S, cnt, first);
            h->stats.kernel_launches += 1;
        } else {
            long long* tot = first + (nw + 1);
            row_total_kernel<<<(nw + 1 + T - 1) / T, T, 0, st>>>(nw, S, cnt, tot);
            SGPR_TRY(scan_exclusive_ll(h, tot, first, nw + 1, st));
            h->stats.kernel_launches += 3;
        }
    }
    long long total = 0;
    if (warm) {
        h->row_first_host_valid = false;
    } else {
        long long part[2] = {0, 0};   // block-per-bin pairs (cursor), warp-kernel pairs
        int err[4] = {0, 0, 0, 0};
        unsigned long long berr[2] = {0, 0};
        int rf[SGPR_MAX_SPECIES + 1];
        SGPR_CUDA(cudaMemcpyAsync(&part[0], cursor, sizeof(long long), cudaMemcpyDeviceToHost, st));
        if (nw > 0) SGPR_CUDA(cudaMemcpyAsync(&part[1], first + nw, sizeof(long long), cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaMemcpyAsync(err, h->errflag.p, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
        if (bg) SGPR_CUDA(cudaMemcpyAsync(berr, bg->err, sizeof(berr), cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaMemcpy2DAsync(rf, sizeof(int), row_first_src, (size_t)row_first_pitch, sizeof(int), S + 1,
                                    cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaStreamSynchronize(st));
        SGPR_TRY(bg ? check_batch_err(berr) : check_err_flags(err));
        for (int s = 0; s <= S; ++s) h->row_first[s] = rf[s];
        h->row_first_host_valid = true;
        total = part[0] + part[1];
        if (total + 1 > h->pairs_cap) {
            const long long want = total + total / 4 + 4096;
            SGPR_TRY(h->nl_pairs.ensure(sizeof(PairRec) * (size_t)want));
            h->pairs_cap = (long long)(h->nl_pairs.bytes / sizeof(PairRec)) - 1;
            if (done > 0) {
                SGPR_CUDA(cudaMemsetAsync(cursor, 0, sizeof(long long), st));
                launch_neighbor_bins(h, g, contig_c0, contig_c0 + done, 0, nullptr, st);
            }
        }
    }
    if (nw > 0) launch_neighbor<true>(h, st, done, nw, g, first, nullptr, bg);
    nl_finish_kernel<<<1, 1024, 0, st>>>(na, S, row_first_src, row_first_pitch / (int)sizeof(int), h->row_first_d.as<int>(),
                                         warm ? 1 : 0, cursor, nw > 0 ? first + nw : nullptr, h->pairs_cap,
                                         h->errflag.as<int>(), h->status_d.as<long long>(), h->nl_rows.as<longlong2>());
    h->stats.kernel_launches += 1;
    SGPR_CUDA(cudaGetLastError());
    *n_pairs = total;
    return SGPR_OK;
}

// Neighbour list of ALL atoms (single-GPU path): rows in cell order, descriptor rows from the species-major scan of
// cell_sort.  Output: nl_rows [N] (begin, end) into nl_pairs, each row ordered by neighbour species, then bin traversal
// order, then cell order; h->row_first.  bg: all atoms of a batch, one warp per environment (batched neighbor_kernel);
// always a sizing step.
int neighbor_build(sgpr_context* h, int64_t N, const Geom& g, cudaStream_t st, int64_t* n_pairs, bool warm,
                   const BatchGeom* bg) {
    h->active_all = true;
    h->n_active = N;
    SGPR_TRY(h->nl_cnt.ensure(sizeof(int) * ((size_t)N * h->S + 1)));
    SGPR_TRY(h->nl_masks.ensure(sizeof(unsigned) * kMaskSlots * ((size_t)N + 1)));
    SGPR_TRY(h->nl_rows.ensure(sizeof(longlong2) * ((size_t)N + 1)));
    launch_count(h, 0, (int)N, g, nullptr, st, 0, bg);
    const int ncell = bg ? bg->ncell : g.ncell;
    const int* rstartT = h->rstart.as<int>() + (ncell * h->S + 1);
    return nl_finish(h, g, st, rstartT, (int)sizeof(int) * ncell, n_pairs, 0, (int)N, warm, bg);
}

// ---------------------------------------------------------------------------------
// atom sharding (SURVEY.md section 8e)
// ---------------------------------------------------------------------------------
__global__ void shard_init_kernel(int64_t N, int c0, int c1, unsigned char* __restrict__ owned,
                                  unsigned char* __restrict__ mark, int* __restrict__ active, int* __restrict__ rowof) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= N) return;
    const bool own = (c >= c0 && c < c1);
    owned[c] = own ? 1 : 0;
    mark[c] = 0;
    rowof[c] = -1;
    if (own) active[c - c0] = (int)c;
}
__global__ void halo_flag_kernel(int64_t N, const unsigned char* __restrict__ owned, const unsigned char* __restrict__ mark,
                                 int* __restrict__ flag) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c > N) return;
    flag[c] = (c < N && mark[c] && !owned[c]) ? 1 : 0;
}
__global__ void halo_scatter_kernel(int64_t N, const int* __restrict__ flag, const int* __restrict__ pos, int n_own,
                                    int* __restrict__ active) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= N) return;
    if (flag[c]) active[n_own + pos[c]] = (int)c;
}
__global__ void species_flag_kernel(int na, const int* __restrict__ active, const AtomRec* __restrict__ atoms, int s,
                                    int* __restrict__ flag) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > na) return;
    flag[k] = (k < na && meta_species(atoms[active[k]].meta) == s) ? 1 : 0;
}
__global__ void species_rows_kernel(int na, const int* __restrict__ active, const AtomRec* __restrict__ atoms, int s,
                                    const int* __restrict__ flag, const int* __restrict__ pos,
                                    int* __restrict__ row_first_d, const unsigned char* __restrict__ owned,
                                    int* __restrict__ rowof, unsigned char* __restrict__ row_owned) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > na) return;
    const int base = row_first_d[s];
    if (k == na) {
        row_first_d[s + 1] = base + pos[na];  // read by the launch for species s+1 (stream order)
        return;
    }
    if (flag[k]) {
        const int c = active[k];
        const int row = base + pos[k];
        rowof[c] = row;
        row_owned[row] = owned[c];
    }
}

// Contiguous owned range [c0, c1) of the cell order (no halo): species-major local rows follow directly from
// the two scans of cell_sort -- count of species-s atoms before a cell index c:
//   before_s(c) = (rstartT[s][bin(c)] - rstartT[s][0]) + clamp(c - cstart[bin(c)][s], 0, cnt[bin(c)][s])
__global__ void contig_species_kernel(int64_t N, int c0, int c1, int S, int ncell, const int* __restrict__ abin,
                                      const int* __restrict__ cstart, const int* __restrict__ rstartT,
                                      int* __restrict__ row_first_d, int* __restrict__ before0) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int acc = 0;
    for (int s = 0; s < S; ++s) {
        int b[2];
        for (int e = 0; e < 2; ++e) {
            const int c = e == 0 ? c0 : c1;
            if (c >= N) {
                b[e] = rstartT[s * ncell + ncell - 1] - rstartT[s * ncell] +
                       (cstart[(ncell - 1) * S + s + 1] - cstart[(ncell - 1) * S + s]);
            } else {
                const int bin = abin[c];
                const int lo = cstart[bin * S + s], hi = cstart[bin * S + s + 1];
                b[e] = rstartT[s * ncell + bin] - rstartT[s * ncell] + max(0, min(c, hi) - lo);
            }
        }
        before0[s] = b[0];
        row_first_d[s] = acc;
        acc += b[1] - b[0];
    }
    row_first_d[S] = acc;
}
__global__ void contig_rows_kernel(int c0, int n_own, int S, int ncell, const AtomRec* __restrict__ atoms,
                                   const int* __restrict__ abin, const int* __restrict__ cstart,
                                   const int* __restrict__ rstartT, const int* __restrict__ row_first_d,
                                   const int* __restrict__ before0, int* __restrict__ rowof,
                                   unsigned char* __restrict__ row_owned) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_own) return;
    const int c = c0 + k;
    const int s = meta_species(atoms[c].meta), bin = abin[c];
    const int global_rank = rstartT[s * ncell + bin] - rstartT[s * ncell] + (c - cstart[bin * S + s]);
    const int row = row_first_d[s] + (global_rank - before0[s]);
    rowof[c] = row;
    row_owned[row] = 1;
}

// Owned range of the cell order + exact one-cutoff halo (atoms that have an owned atom as a
// neighbour).  Active list = owned ++ halo; rows are species-major over the active list.
int neighbor_build_sharded(sgpr_context* h, int64_t N, const Geom& g, int rank, int world, cudaStream_t st,
                           int64_t* n_pairs, bool with_halo, bool warm) {
    if (warm && with_halo) {
        set_error("internal: the halo mode sizes its active list on the host");
        return SGPR_ERR_INVALID;
    }
    const int S = h->S;
    const int c0 = (int)((N * rank) / world), c1 = (int)((N * (rank + 1)) / world);
    const int n_own = c1 - c0;
    h->active_all = false;
    h->n_owned = n_own;
    SGPR_TRY(h->owned.ensure(2 * ((size_t)N + 1)));
    SGPR_TRY(h->active_list.ensure(sizeof(int) * ((size_t)N + 1)));
    SGPR_TRY(h->shard_tmp.ensure(sizeof(int) * (2 * ((size_t)N + 2) + 2 * SGPR_MAX_SPECIES + 4)));
    SGPR_TRY(h->row_owned.ensure((size_t)N + 1));
    SGPR_TRY(h->nl_cnt.ensure(sizeof(int) * ((size_t)N * S + 1)));
    SGPR_TRY(h->nl_masks.ensure(sizeof(unsigned) * kMaskSlots * ((size_t)N + 1)));
    unsigned char* owned = h->owned.as<unsigned char>();
    unsigned char* mark = owned + (N + 1);
    int* active = h->active_list.as<int>();
    int* flag = h->shard_tmp.as<int>();
    int* pos = flag + (N + 2);
    int* row_first_d = pos + (N + 2);
    int* rowof = h->rowof.as<int>() + (N + 1);
    const int T = 256;
    const int nblkN = (int)((N + 1 + T - 1) / T);
    shard_init_kernel<<<nblkN, T, 0, st>>>(N, c0, c1, owned, mark, active, rowof);
    h->n_active = n_own;
    SGPR_TRY(h->nl_rows.ensure(sizeof(longlong2) * ((size_t)N + 1)));
    launch_count(h, 0, n_own, g, with_halo ? mark : nullptr, st, c0);
    int n_halo = 0;
    if (with_halo) {
        halo_flag_kernel<<<nblkN, T, 0, st>>>(N, owned, mark, flag);
        size_t tmp = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tmp, flag, pos, (int)N + 1, st);
        SGPR_TRY(h->scan_tmp.ensure(tmp));
        SGPR_CUDA(cub::DeviceScan::ExclusiveSum(h->scan_tmp.p, tmp, flag, pos, (int)N + 1, st));
        halo_scatter_kernel<<<nblkN, T, 0, st>>>(N, flag, pos, n_own, active);
        SGPR_CUDA(cudaMemcpyAsync(&n_halo, pos + N, sizeof(int), cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaStreamSynchronize(st));
    }
    const int na = n_own + n_halo;
    h->n_active = na;
    launch_count(h, n_own, n_halo, g, nullptr, st, -1);
    // species-major rows over the active list
    SGPR_CUDA(cudaMemsetAsync(row_first_d, 0, sizeof(int) * (SGPR_MAX_SPECIES + 1), st));
    const int nblkA = (na + 1 + T - 1) / T;
    if (!with_halo) {
        // contiguous active set: two small kernels instead of S x (flag, scan, assign)
        const int nkeys = g.ncell * S;
        const int* rstartT = h->rstart.as<int>() + (nkeys + 1);
        int* before0 = row_first_d + SGPR_MAX_SPECIES + 1;
        contig_species_kernel<<<1, 32, 0, st>>>(N, c0, c1, S, g.ncell, h->rowof.as<int>(), h->cstart.as<int>(), rstartT,
                                                row_first_d, before0);
        if (n_own > 0)
            contig_rows_kernel<<<(n_own + T - 1) / T, T, 0, st>>>(c0, n_own, S, g.ncell, h->atoms.as<AtomRec>(),
                                                                 h->rowof.as<int>(), h->cstart.as<int>(), rstartT,
                                                                 row_first_d, before0, rowof,
                                                                 h->row_owned.as<unsigned char>());
        h->stats.kernel_launches += 3;
        SGPR_CUDA(cudaGetLastError());
        return nl_finish(h, g, st, row_first_d, (int)sizeof(int), n_pairs, c0, n_own, warm);
    }
    for (int s = 0; s < S; ++s) {
        species_flag_kernel<<<nblkA, T, 0, st>>>(na, active, h->atoms.as<AtomRec>(), s, flag);
        size_t tmp = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tmp, flag, pos, na + 1, st);
        SGPR_TRY(h->scan_tmp.ensure(tmp));
        SGPR_CUDA(cub::DeviceScan::ExclusiveSum(h->scan_tmp.p, tmp, flag, pos, na + 1, st));
        species_rows_kernel<<<nblkA, T, 0, st>>>(na, active, h->atoms.as<AtomRec>(), s, flag, pos, row_first_d, owned,
                                                 rowof, h->row_owned.as<unsigned char>());
    }
    h->stats.kernel_launches += 5 + 4 * S;
    SGPR_CUDA(cudaGetLastError());
    return nl_finish(h, g, st, row_first_d, (int)sizeof(int), n_pairs, c0, n_own, false);
}

}  // namespace sgpr
