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

__global__ void bin_count_kernel(int64_t N, const double* __restrict__ pos, const int32_t* __restrict__ Z,
                                 const int* __restrict__ ztab, Geom g, int S, int* __restrict__ cnt,
                                 int* __restrict__ key_out, int* __restrict__ rank_out, int* __restrict__ err) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    int z = Z[i];
    int s = (z >= 0 && z < 128) ? ztab[z] : -1;
    if (s < 0) {
        atomicExch(&err[0], 1);
        atomicExch(&err[1], z);
        s = 0;
    }
    int b[3], w[3];
    frac_bin(g, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], b, w);
    if (abs(w[0]) > 120 || abs(w[1]) > 120 || abs(w[2]) > 120) atomicExch(&err[0], 2);
    int bin = (b[0] * g.nb[1] + b[1]) * g.nb[2] + b[2];
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

// one thread per key: sort the (short) run by original index -> deterministic cell order
__global__ void sort_runs_kernel(int nkeys, const int* __restrict__ cstart, int* __restrict__ order) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nkeys) return;
    int b = cstart[k], e = cstart[k + 1];
    for (int i = b + 1; i < e; ++i) {
        int v = order[i];
        int j = i - 1;
        while (j >= b && order[j] > v) {
            order[j + 1] = order[j];
            --j;
        }
        order[j + 1] = v;
    }
}

__global__ void gather_atoms_kernel(int64_t N, const double* __restrict__ pos, const int* __restrict__ key,
                                    const int* __restrict__ order, const int* __restrict__ cstart,
                                    const int* __restrict__ rstartT, Geom g, int S, AtomRec* __restrict__ atoms,
                                    int* __restrict__ abin, int* __restrict__ rowof) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= N) return;
    int i = order[c];
    int k = key[i];
    int bin = k / S, s = k - bin * S;
    double x = pos[3 * (int64_t)i], y = pos[3 * (int64_t)i + 1], z = pos[3 * (int64_t)i + 2];
    int b[3], w[3];
    frac_bin(g, x, y, z, b, w);
    AtomRec r;
    r.x = x;
    r.y = y;
    r.z = z;
    r.meta = (unsigned long long)(unsigned int)i | ((unsigned long long)s << 32) |
             ((unsigned long long)(w[0] + 128) << 40) | ((unsigned long long)(w[1] + 128) << 48) |
             ((unsigned long long)(w[2] + 128) << 56);
    atoms[c] = r;
    abin[c] = bin;
    rowof[c] = rstartT[s * g.ncell + bin] + (int)(c - cstart[k]);
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
// ranks; the cell order must not depend on them) and write the cell-ordered atom records of the bin.
__global__ void sort_gather_kernel(int ncell, int64_t N, const double* __restrict__ pos, const int* __restrict__ cstart,
                                   const int* __restrict__ rstartT, Geom g, int S, int* __restrict__ order,
                                   AtomRec* __restrict__ atoms, int* __restrict__ abin, int* __restrict__ rowof) {
    const int lane = threadIdx.x & 31;
    const int bin = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (bin >= ncell) return;
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
            AtomRec r;
            r.x = x;
            r.y = y;
            r.z = z;
            r.meta = (unsigned long long)(unsigned int)i | ((unsigned long long)s << 32) |
                     ((unsigned long long)(w[0] + 128) << 40) | ((unsigned long long)(w[1] + 128) << 48) |
                     ((unsigned long long)(w[2] + 128) << 56);
            atoms[c] = r;
            abin[c] = bin;
            rowof[c] = row0 + (c - b);
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
//   rstart  [2*(nkeys+1)]  transposed counts, then their scan: first row of (species, bin)
//   keyrank [2N]        key per original atom, arbitrary rank within key
//   order   [N]         original index of cell-order atom c
//   atoms   [N] AtomRec ; rowof [2N]: abin[c], rowof[c]
//   misc    [16] ints   err flag(2) ...
int cell_sort(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const Geom& g, cudaStream_t st) {
    const int S = h->S;
    const int nkeys = g.ncell * S;
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
    SGPR_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * (nkeys + 1), st));
    SGPR_CUDA(cudaMemsetAsync(err, 0, sizeof(int) * 4, st));
    const int T = 256;
    const int nblkN = (int)((N + T - 1) / T);
    const int nblkK = (nkeys + T - 1) / T;
    if (N > 0)
        bin_count_kernel<<<nblkN, T, 0, st>>>(N, pos_d, Z_d, h->ztab.as<int>(), g, S, cnt, key, rank, err);
    if (h->nl_lean && nkeys + 1 <= kScanMaxKeys) {
        // lean path (< 2^18 bin x species keys): 4 kernels instead of 9
        key_scan_kernel<<<2, kScanThreads, 0, st>>>(nkeys, g.ncell, S, cnt, cstart, rstartT);
        if (N > 0) {
            scatter_order_kernel<<<nblkN, T, 0, st>>>(N, key, rank, cstart, h->order.as<int>());
            sort_gather_kernel<<<(g.ncell + 7) / 8, 256, 0, st>>>(g.ncell, N, pos_d, cstart, rstartT, g, S, h->order.as<int>(),
                                                               h->atoms.as<AtomRec>(), h->rowof.as<int>(),
                                                               h->rowof.as<int>() + (N + 1));
        }
        h->stats.kernel_launches += 4;
        SGPR_CUDA(cudaGetLastError());
        return SGPR_OK;
    }
    SGPR_CUDA(cudaMemsetAsync(cntT, 0, sizeof(int) * (nkeys + 1), st));
    transpose_cnt_kernel<<<nblkK, T, 0, st>>>(g.ncell, S, cnt, cntT);
    SGPR_TRY(scan_exclusive_int(h, cnt, cstart, nkeys + 1, st));
    SGPR_TRY(scan_exclusive_int(h, cntT, rstartT, nkeys + 1, st));
    if (N > 0) {
        scatter_order_kernel<<<nblkN, T, 0, st>>>(N, key, rank, cstart, h->order.as<int>());
        sort_runs_kernel<<<nblkK, T, 0, st>>>(nkeys, cstart, h->order.as<int>());
        gather_atoms_kernel<<<nblkN, T, 0, st>>>(N, pos_d, key, h->order.as<int>(), cstart, rstartT, g, S,
                                                 h->atoms.as<AtomRec>(), h->rowof.as<int>(),
                                                 h->rowof.as<int>() + (N + 1));
    }
    h->stats.kernel_launches += 9;  // 5 own kernels + 2 cub scans (2 kernels each)
    SGPR_CUDA(cudaGetLastError());
    return SGPR_OK;
}

// ---------------------------------------------------------------------------------
// cell sort of a batch: keys (bin_base[b] + bin) * S + species -- structure-major, so every structure is one contiguous
// range of the cell order and of each species' rows, and the second (species-major) scan still gives one row block per
// central species for the whole batch
// ---------------------------------------------------------------------------------
// structure of atom i: the last b with first[b] <= i (empty structures are skipped)
__device__ __forceinline__ int batch_of(const long long* __restrict__ first, int B, long long i) {
    int lo = 0, hi = B;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (first[mid] <= i) lo = mid;
        else hi = mid;
    }
    return lo;
}

__global__ void batch_bin_count_kernel(int64_t N, const double* __restrict__ pos, const int32_t* __restrict__ Z,
                                       const int* __restrict__ ztab, BatchGeom bg, int S, int* __restrict__ cnt,
                                       int* __restrict__ key_out, int* __restrict__ rank_out) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int b = batch_of(bg.first, bg.B, i);
    int z = Z[i];
    int s = (z >= 0 && z < 128) ? ztab[z] : -1;
    if (s < 0) {
        atomicMin(&bg.err[0], ((unsigned long long)b << 32) | (unsigned)z);
        s = 0;
    }
    int bn[3], w[3];
    frac_bin(bg.geoms[b], pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], bn, w);
    if (abs(w[0]) > 120 || abs(w[1]) > 120 || abs(w[2]) > 120) atomicMin(&bg.err[1], (unsigned long long)b);
    const Geom& g = bg.geoms[b];
    int bin = bg.bin_base[b] + (bn[0] * g.nb[1] + bn[1]) * g.nb[2] + bn[2];
    int key = bin * S + s;
    key_out[i] = key;
    rank_out[i] = atomicAdd(&cnt[key], 1);
}

// cell-ordered atom records (runs already sorted by original index), global bin, row, structure
__global__ void batch_gather_kernel(int64_t N, const double* __restrict__ pos, const int* __restrict__ key,
                                    const int* __restrict__ order, const int* __restrict__ cstart,
                                    const int* __restrict__ rstartT, BatchGeom bg, int S, AtomRec* __restrict__ atoms,
                                    int* __restrict__ abin, int* __restrict__ rowof) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= N) return;
    int i = order[c];
    int k = key[i];
    int bin = k / S, s = k - bin * S;
    const int b = batch_of(bg.first, bg.B, i);
    double x = pos[3 * (int64_t)i], y = pos[3 * (int64_t)i + 1], z = pos[3 * (int64_t)i + 2];
    int b3[3], w[3];
    frac_bin(bg.geoms[b], x, y, z, b3, w);
    AtomRec r;
    r.x = x;
    r.y = y;
    r.z = z;
    r.meta = (unsigned long long)(unsigned int)i | ((unsigned long long)s << 32) |
             ((unsigned long long)(w[0] + 128) << 40) | ((unsigned long long)(w[1] + 128) << 48) |
             ((unsigned long long)(w[2] + 128) << 56);
    atoms[c] = r;
    abin[c] = bin;
    rowof[c] = rstartT[s * bg.ncell + bin] + (int)(c - cstart[k]);
    bg.astr[c] = b;
}

// Same workspace layout as cell_sort, plus h->astr.  Errors are reported by batch_neighbor_build's sizing step.
int batch_cell_sort(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const BatchGeom& bg, cudaStream_t st) {
    const int S = h->S;
    const int nkeys = bg.ncell * S;
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
    SGPR_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * (nkeys + 1), st));
    SGPR_CUDA(cudaMemsetAsync(h->errflag.p, 0, sizeof(int) * 4, st));
    SGPR_CUDA(cudaMemsetAsync(bg.err, 0x7f, sizeof(unsigned long long) * 2, st));
    const int T = 256;
    const int nblkN = (int)((N + T - 1) / T);
    const int nblkK = (nkeys + T - 1) / T;
    if (N > 0) batch_bin_count_kernel<<<nblkN, T, 0, st>>>(N, pos_d, Z_d, h->ztab.as<int>(), bg, S, cnt, key, rank);
    if (nkeys + 1 <= kScanMaxKeys) {
        key_scan_kernel<<<2, kScanThreads, 0, st>>>(nkeys, bg.ncell, S, cnt, cstart, rstartT);
    } else {
        SGPR_CUDA(cudaMemsetAsync(cntT, 0, sizeof(int) * (nkeys + 1), st));
        transpose_cnt_kernel<<<nblkK, T, 0, st>>>(bg.ncell, S, cnt, cntT);
        SGPR_TRY(scan_exclusive_int(h, cnt, cstart, nkeys + 1, st));
        SGPR_TRY(scan_exclusive_int(h, cntT, rstartT, nkeys + 1, st));
    }
    if (N > 0) {
        scatter_order_kernel<<<nblkN, T, 0, st>>>(N, key, rank, cstart, h->order.as<int>());
        sort_runs_kernel<<<nblkK, T, 0, st>>>(nkeys, cstart, h->order.as<int>());
        batch_gather_kernel<<<nblkN, T, 0, st>>>(N, pos_d, key, h->order.as<int>(), cstart, rstartT, bg, S,
                                                 h->atoms.as<AtomRec>(), h->rowof.as<int>(), h->rowof.as<int>() + (N + 1));
    }
    h->stats.kernel_launches += 5;
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
// the geometry an environment's search uses: the call's, or (batch) that of the centre's structure
template <bool BATCH>
__device__ __forceinline__ const Geom& env_geom(const Geom& g, const BatchGeom& bg, int b) {
    if constexpr (BATCH)
        return bg.geoms[b];
    else
        return g;
}

// BATCH: a batch of structures (sgpr_predict_batch) -- each environment reads its structure's Geom, and its stencil
// stays inside that structure's bins (bg.bin_base); same traversal, pair_test and pair order as a call on the structure
template <bool FILL, int NS, bool BATCH = false>
__global__ void __launch_bounds__(256) neighbor_kernel(int env0, int n_env, const int* __restrict__ active,
                                                       const AtomRec* __restrict__ atoms, const int* __restrict__ abin,
                                                       const int* __restrict__ cstart, Geom g_call, int S,
                                                       int* __restrict__ nl_cnt, const long long* __restrict__ nl_first,
                                                       PairRec* __restrict__ pairs, unsigned char* __restrict__ mark,
                                                       unsigned* __restrict__ masks, BatchGeom bg = BatchGeom{}) {
    const int lane = threadIdx.x & 31;
    int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (wid >= n_env) return;
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
    if (FILL) {
        long long o = nl_first[wid];
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            base[s] = o;
            if (s < S) o += nl_cnt[(long long)wid * S + s];
        }
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
                            if (acc && sp == s) {
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
// neighbour search, one BLOCK per bin (the path for all but tiny systems): every atom of a bin walks the
// same stencil, so the block gathers the candidates of the stencil once into shared memory -- already
// shifted to the right periodic image -- and its warps then test their atoms against that tile without
// touching global memory.  Same two passes, masks, pair order and exact accept rule as neighbor_kernel:
// the shared-memory test decides everything except d^2 within 1e-11 of rc^2, which goes through
// pair_test (the reference's rounding sequence).
// ---------------------------------------------------------------------------------
constexpr int kBinThreads = 256, kBinCap = 1024, kRunChunk = 128;

template <bool FILL, int NS>
__global__ void __launch_bounds__(kBinThreads, 4) neighbor_bin_kernel(int c_begin, int c_end, int env0,
                                                                   const AtomRec* __restrict__ atoms,
                                                                   const int* __restrict__ cstart, Geom g, int S,
                                                                   int* __restrict__ nl_cnt,
                                                                   const long long* __restrict__ nl_first,
                                                                   PairRec* __restrict__ pairs, unsigned char* __restrict__ mark,
                                                                   unsigned* __restrict__ masks, int* __restrict__ nl_run) {
    // candidate image relative to the bin's first atom, in float (x, y, z), and w = |x| + |y| + |z| of the unshifted and
    // shifted absolute coordinates (rounding bound of the double-precision test)
    __shared__ float4 rel[kBinCap];
    __shared__ unsigned maxabs_u;            // running max of the relative coordinates' 1-norm (float bits)
    __shared__ int pj[kBinCap];
    __shared__ unsigned code[kBinCap];       // bin shift (3 x int8) | species << 24
    __shared__ int run_beg[kRunChunk], run_pre[kRunChunk + 1];
    __shared__ unsigned run_sh[kRunChunk];
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
    int slot_base = 0, tile_no = 0;
    for (int r0 = 0; r0 < nruns; r0 += kRunChunk) {
        const int nr = min(kRunChunk, nruns - r0);
        __syncthreads();
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
        const int total = run_pre[nr];
        for (int t0 = 0; t0 < total; t0 += kBinCap) {
            const int n = min(kBinCap, total - t0);
            const bool last_tile = (r0 + kRunChunk >= nruns) && (t0 + kBinCap >= total);
            if (t0 > 0) __syncthreads();   // the previous tile is still being read
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
            }
            {
                const unsigned m = __reduce_max_sync(0xffffffffu, __float_as_uint(my_max));   // floats >= 0 order as uints
                if (lane == 0 && m > 0u) atomicMax(&maxabs_u, m);
            }
            __syncthreads();
            const float maxabs = __uint_as_float(maxabs_u);
            // accept bits of an environment: one 64-bit word per lane, bit k = candidate (slot k, this lane)
            const int nb_tile = (n + 31) >> 5;
            const int nb_masked = max(0, min(nb_tile, kMaskSlots - slot_base));   // batches of this tile covered by the word
            for (int c = lo + warp; c < hi; c += NW) {
                const int wid = c - c_begin + env0;
                const AtomRec ai = atoms[c];
                unsigned long long* my_word = reinterpret_cast<unsigned long long*>(masks) + (size_t)wid * 32 + lane;
                unsigned long long accw = 0ull;
                long long first_pair = 0;
                int cnt_s[NS];
                if (FILL) {
                    accw = *my_word;
                    first_pair = nl_first[wid];
#pragma unroll
                    for (int s = 0; s < NS; ++s) cnt_s[s] = s < S ? nl_cnt[(long long)wid * S + s] : 0;
                } else if (tile_no > 0 && slot_base < kMaskSlots) {
                    accw = *my_word;
                }
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
                auto test = [&](int q) -> bool {
                    const float4 cq = rel[q];
                    const float ex = cq.x - fxi, ey = cq.y - fyi, ez = cq.z - fzi;
                    const float d2f = fmaf(ex, ex, fmaf(ey, ey, ez * ez));
                    if (d2f > hi_f) return false;
                    if (d2f < lo_f && d2f > margin) return true;
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
                if (!FILL) {
                    unsigned long long pc0 = 0ull, pc1 = 0ull;   // packed per-lane counters, 16 bits per species
                    for (int b = 0; b < nb_tile; ++b) {
                        const int q = b * 32 + lane;
                        if (q < n && test(q)) {
                            const int sp = (int)(code[q] >> 24);
                            if (mark) mark[pj[q]] = 1;   // atoms whose environment the owner needs (halo)
                            const unsigned long long one = 1ull << (16 * (sp & 3));
                            if (NS <= 4 || sp < 4) pc0 += one;
                            else pc1 += one;
                            if (b < nb_masked) accw |= 1ull << (slot_base + b);
                        }
                    }
                    if (nb_masked > 0) *my_word = accw;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        pc0 += __shfl_xor_sync(0xffffffffu, pc0, o);
                        if (NS > 4) pc1 += __shfl_xor_sync(0xffffffffu, pc1, o);
                    }
                    if (lane == 0) {
#pragma unroll
                        for (int s = 0; s < NS; ++s)
                            if (s < S) {
                                const int v = (int)(((s < 4 ? pc0 : pc1) >> (16 * (s & 3))) & 0xffffull);
                                int* dst = nl_cnt + (long long)wid * S + s;
                                *dst = tile_no > 0 ? *dst + v : v;
                            }
                    }
                } else {
                    // pairs of one species are contiguous; inside a species: tile, then lane, then slot
                    long long start[NS];
                    {
                        long long o = first_pair;
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            start[s] = o + ((tile_no > 0 && s < S) ? nl_run[(long long)wid * S + s] : 0);
                            o += cnt_s[s];
                        }
                    }
                    auto emit = [&](int q, unsigned long long& run0, unsigned long long& run1) {
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
                    // this lane's accepted candidates of the tile: stored bits, recomputed beyond the word's reach
                    unsigned long long wt = nb_masked > 0 ? (accw >> slot_base) : 0ull;
                    if (nb_masked < 64) wt &= (1ull << nb_masked) - 1ull;
                    unsigned long long pc0 = 0ull, pc1 = 0ull;
                    for (unsigned long long t = wt; t; t &= t - 1) {
                        const int sp = (int)(code[(__ffsll((long long)t) - 1) * 32 + lane] >> 24);
                        const unsigned long long one = 1ull << (16 * (sp & 3));
                        if (NS <= 4 || sp < 4) pc0 += one;
                        else pc1 += one;
                    }
                    for (int b = nb_masked; b < nb_tile; ++b) {   // rare: more than kMaskSlots batches
                        const int q = b * 32 + lane;
                        if (q < n && test(q)) {
                            const int sp = (int)(code[q] >> 24);
                            const unsigned long long one = 1ull << (16 * (sp & 3));
                            if (NS <= 4 || sp < 4) pc0 += one;
                            else pc1 += one;
                        }
                    }
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
                    for (unsigned long long t = wt; t; t &= t - 1) emit((__ffsll((long long)t) - 1) * 32 + lane, run0, run1);
                    for (int b = nb_masked; b < nb_tile; ++b) {
                        const int q = b * 32 + lane;
                        if (q < n && test(q)) emit(q, run0, run1);
                    }
                    if (!last_tile && lane == 0) {
#pragma unroll
                        for (int s = 0; s < NS; ++s)
                            if (s < S) {
                                const int prev = tile_no > 0 ? nl_run[(long long)wid * S + s] : 0;
                                nl_run[(long long)wid * S + s] = prev + (int)(((s < 4 ? tot0 : tot1) >> (16 * (s & 3))) & 0xffffull);
                            }
                    }
                }
            }
            slot_base += (n + 31) >> 5;
            ++tile_no;
        }
    }
}

template <bool FILL>
static void launch_neighbor_bins(cudaStream_t st, int S, int c_begin, int c_end, int env0, const AtomRec* atoms,
                                 const int* cstart, const Geom& g, int* nl_cnt, const long long* nl_first, PairRec* pairs,
                                 unsigned char* mark, unsigned* masks, int* nl_run) {
    const int nblk = g.ncell, T = kBinThreads;
    if (S <= 1)
        neighbor_bin_kernel<FILL, 1><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, nl_run);
    else if (S <= 2)
        neighbor_bin_kernel<FILL, 2><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, nl_run);
    else if (S <= 4)
        neighbor_bin_kernel<FILL, 4><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, nl_run);
    else
        neighbor_bin_kernel<FILL, 8><<<nblk, T, 0, st>>>(c_begin, c_end, env0, atoms, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, nl_run);
}

// the block-per-bin kernels need enough bins to fill the machine; tiny systems keep one warp per environment
static bool use_bin_kernels(const sgpr_context* h, const Geom& g) { return h->nl_mode == 2 || (g.ncell >= 64 && h->nl_mode != 1); }

template <bool FILL>
static void launch_neighbor(int nblk, int T, cudaStream_t st, int S, int env0, int n_env, const int* active,
                            const AtomRec* atoms, const int* abin, const int* cstart, const Geom& g, int* nl_cnt,
                            const long long* nl_first, PairRec* pairs, unsigned char* mark, unsigned* masks,
                            const BatchGeom* bg = nullptr) {
    if (bg) {
        if (S <= 1)
            neighbor_kernel<FILL, 1, true><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, *bg);
        else if (S <= 2)
            neighbor_kernel<FILL, 2, true><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, *bg);
        else if (S <= 4)
            neighbor_kernel<FILL, 4, true><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, *bg);
        else
            neighbor_kernel<FILL, 8, true><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks, *bg);
        return;
    }
    if (S <= 1)
        neighbor_kernel<FILL, 1><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks);
    else if (S <= 2)
        neighbor_kernel<FILL, 2><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks);
    else if (S <= 4)
        neighbor_kernel<FILL, 4><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks);
    else
        neighbor_kernel<FILL, 8><<<nblk, T, 0, st>>>(env0, n_env, active, atoms, abin, cstart, g, S, nl_cnt, nl_first, pairs, mark, masks);
}

__global__ void row_total_kernel(int n, int S, const int* __restrict__ nl_cnt, long long* __restrict__ tot) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    long long t = 0;
    if (i < n)
        for (int s = 0; s < S; ++s) t += nl_cnt[(long long)i * S + s];
    tot[i] = t;
}

// contig_c0 >= 0: environments env0 .. env0+n_env-1 are the atoms contig_c0 .. of the cell order
static int launch_count(sgpr_context* h, int env0, int n_env, const Geom& g, unsigned char* mark, cudaStream_t st,
                        int contig_c0, const BatchGeom* bg = nullptr) {
    if (n_env <= 0) return SGPR_OK;
    if (contig_c0 >= 0 && !bg && use_bin_kernels(h, g)) {
        launch_neighbor_bins<false>(st, h->S, contig_c0, contig_c0 + n_env, env0, h->atoms.as<AtomRec>(), h->cstart.as<int>(), g,
                                    h->nl_cnt.as<int>(), nullptr, nullptr, mark, h->nl_masks.as<unsigned>(), nullptr);
        h->stats.kernel_launches += 1;
        return SGPR_OK;
    }
    const int T = 256;
    const int nblk = (int)(((int64_t)n_env * 32 + T - 1) / T);
    launch_neighbor<false>(nblk, T, st, h->S, env0, n_env, h->active_all ? nullptr : h->active_list.as<int>(),
                           h->atoms.as<AtomRec>(), h->rowof.as<int>(), h->cstart.as<int>(), g, h->nl_cnt.as<int>(), nullptr,
                           nullptr, mark, h->nl_masks.as<unsigned>(), bg);
    h->stats.kernel_launches += 1;
    return SGPR_OK;
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

// batch errors name the first structure that failed (batch_bin_count_kernel)
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

// Sync-free steps: the pair count and the error flags stay on the device.  One thread records them in the status
// block and decides whether the step is valid (the pair list fits the capacity sized by an earlier step, no error
// flag); an invalid step gets EMPTY neighbour rows, so that every later kernel stays inside its buffers -- the step's
// results are then meaningless and the sticky counter status[1] says so (sgpr_check / the host entry point re-run it).
__global__ void nl_status_kernel(int na, const long long* __restrict__ first, long long cap, const int* __restrict__ err,
                                 long long* __restrict__ status) {
    const long long total = first[na];
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
}
__global__ void nl_clamp_kernel(int na, long long* __restrict__ first, const long long* __restrict__ status) {
    if (status[6] == 0) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= na) first[i] = 0;
}

// Lean form of row totals -> exclusive scan -> species row ranges -> (sync-free steps) status + clamp: one block walks the
// rows in coalesced tiles of 1024 with a running carry.  (A few microseconds for 1e5 rows, and one graph node instead of
// six: what matters for small systems and for the per-rank share of a sharded one.)
constexpr int kRowsScanMax = 1 << 16;   // beyond: row_total + cub scan + status + clamp (one SM would be the bottleneck)
__global__ void __launch_bounds__(1024) rows_scan_kernel(int na, int S, const int* __restrict__ nl_cnt,
                                                         long long* __restrict__ first, const int* __restrict__ row_first_src,
                                                         int row_first_pitch_ints, int* __restrict__ row_first_d, int do_status,
                                                         long long cap, const int* __restrict__ err,
                                                         long long* __restrict__ status) {
    __shared__ int bad_s;
    if ((int)threadIdx.x <= S) row_first_d[threadIdx.x] = row_first_src[(size_t)threadIdx.x * row_first_pitch_ints];
    const long long total = block_scan_exclusive<long long>(
        na + 1,
        [&](int i) -> long long {
            if (i >= na) return 0;
            if (S == 4) {
                const int4 c = *reinterpret_cast<const int4*>(nl_cnt + 4 * (long long)i);
                return (long long)c.x + c.y + c.z + c.w;
            }
            long long t = 0;
            for (int s = 0; s < S; ++s) t += nl_cnt[(long long)i * S + s];
            return t;
        },
        [&](int i, long long v) { first[i] = v; });
    if (!do_status) return;
    if (threadIdx.x == 0) {
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
        for (int i = threadIdx.x; i <= na; i += 1024) first[i] = 0;
}

// row totals -> exclusive scan -> (sizing step: sync for pair count, error flags, species row ranges) -> fill
static int nl_finish(sgpr_context* h, const Geom& g, cudaStream_t st, const int* row_first_src, int row_first_pitch,
                     int64_t* n_pairs, int contig_c0, int n_contig, bool warm, const BatchGeom* bg = nullptr) {
    const int S = h->S;
    const int na = (int)h->n_active;
    SGPR_TRY(h->nl_first.ensure(sizeof(long long) * 2 * ((size_t)na + 1)));
    SGPR_TRY(h->row_first_d.ensure(sizeof(int) * (SGPR_MAX_SPECIES + 2)));
    SGPR_TRY(h->status_d.ensure(sizeof(long long) * 8));
    long long* first = h->nl_first.as<long long>();
    long long* tot = first + (na + 1);
    const int T = 256;
    const bool lean = h->nl_lean && na + 1 <= kRowsScanMax && row_first_pitch % (int)sizeof(int) == 0;
    if (lean) {
        rows_scan_kernel<<<1, 1024, 0, st>>>(na, S, h->nl_cnt.as<int>(), first, row_first_src,
                                             row_first_pitch / (int)sizeof(int), h->row_first_d.as<int>(), warm ? 1 : 0,
                                             h->pairs_cap, h->errflag.as<int>(), h->status_d.as<long long>());
        h->stats.kernel_launches += 1;
    } else {
        row_total_kernel<<<(na + 1 + T - 1) / T, T, 0, st>>>(na, S, h->nl_cnt.as<int>(), tot);
        SGPR_TRY(scan_exclusive_ll(h, tot, first, na + 1, st));
        // species row ranges in their canonical device location (read by the GEMM set-up kernel and row_energy_kernel)
        SGPR_CUDA(cudaMemcpy2DAsync(h->row_first_d.p, sizeof(int), row_first_src, (size_t)row_first_pitch, sizeof(int), S + 1,
                                    cudaMemcpyDeviceToDevice, st));
    }
    long long total = 0;
    if (warm) {
        h->row_first_host_valid = false;
        if (!lean) {
            nl_status_kernel<<<1, 1, 0, st>>>(na, first, h->pairs_cap, h->errflag.as<int>(), h->status_d.as<long long>());
            nl_clamp_kernel<<<(na + 1 + T - 1) / T, T, 0, st>>>(na, first, h->status_d.as<long long>());
            h->stats.kernel_launches += 2;
        }
    } else {
        int err[4] = {0, 0, 0, 0};
        unsigned long long berr[2] = {0, 0};
        int rf[SGPR_MAX_SPECIES + 1];
        SGPR_CUDA(cudaMemcpyAsync(&total, first + na, sizeof(long long), cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaMemcpyAsync(err, h->errflag.p, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
        if (bg) SGPR_CUDA(cudaMemcpyAsync(berr, bg->err, sizeof(berr), cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaMemcpy2DAsync(rf, sizeof(int), row_first_src, (size_t)row_first_pitch, sizeof(int), S + 1,
                                    cudaMemcpyDeviceToHost, st));
        SGPR_CUDA(cudaStreamSynchronize(st));
        SGPR_TRY(bg ? check_batch_err(berr) : check_err_flags(err));
        for (int s = 0; s <= S; ++s) h->row_first[s] = rf[s];
        h->row_first_host_valid = true;
        // capacity with head room: the following steps of a trajectory reuse it without asking the device
        if (total + 1 > h->pairs_cap) {
            const long long want = total + total / 4 + 4096;
            SGPR_TRY(h->nl_pairs.ensure(sizeof(PairRec) * (size_t)want));
            h->pairs_cap = (long long)(h->nl_pairs.bytes / sizeof(PairRec)) - 1;
        }
    }
    int done = 0;   // environments 0 .. n_contig-1 are a contiguous range of the cell order: block-per-bin fill
    if (n_contig > 0 && !bg && use_bin_kernels(h, g)) {
        SGPR_TRY(h->nl_run.ensure(sizeof(int) * ((size_t)n_contig * S + 1)));
        launch_neighbor_bins<true>(st, S, contig_c0, contig_c0 + n_contig, 0, h->atoms.as<AtomRec>(), h->cstart.as<int>(), g,
                                   h->nl_cnt.as<int>(), first, h->nl_pairs.as<PairRec>(), nullptr,
                                   h->nl_masks.as<unsigned>(), h->nl_run.as<int>());
        done = n_contig;
    }
    if (na > done) {
        const int nblk = (int)(((int64_t)(na - done) * 32 + T - 1) / T);
        launch_neighbor<true>(nblk, T, st, S, done, na - done, h->active_all ? nullptr : h->active_list.as<int>(),
                              h->atoms.as<AtomRec>(), h->rowof.as<int>(), h->cstart.as<int>(), g, h->nl_cnt.as<int>(), first,
                              h->nl_pairs.as<PairRec>(), nullptr, h->nl_masks.as<unsigned>(), bg);
    }
    h->stats.kernel_launches += lean ? 1 : 4;  // fill (+ row totals, cub scan (2) when not the one-kernel scan)
    SGPR_CUDA(cudaGetLastError());
    *n_pairs = total;
    return SGPR_OK;
}

// Neighbour list of ALL atoms (single-GPU path): rows in cell order, descriptor rows from the
// species-major scan of cell_sort.  Output: nl_cnt [N,S], nl_first [N+1] (int64), nl_pairs,
// rows ordered by neighbour species, then bin traversal order, then cell order; h->row_first.
int neighbor_build(sgpr_context* h, int64_t N, const Geom& g, cudaStream_t st, int64_t* n_pairs, bool warm) {
    h->active_all = true;
    h->n_active = N;
    SGPR_TRY(h->nl_cnt.ensure(sizeof(int) * ((size_t)N * h->S + 1)));
    SGPR_TRY(h->nl_masks.ensure(sizeof(unsigned) * kMaskSlots * ((size_t)N + 1)));
    SGPR_TRY(launch_count(h, 0, (int)N, g, nullptr, st, 0));
    const int nkeys = g.ncell * h->S;
    const int* rstartT = h->rstart.as<int>() + (nkeys + 1);
    return nl_finish(h, g, st, rstartT, (int)sizeof(int) * g.ncell, n_pairs, 0, (int)N, warm);
}

// Neighbour list of all atoms of a batch: one warp per environment (batched neighbor_kernel), rows in the batch's cell
// order, species row ranges from batch_cell_sort's species-major scan.  Always a sizing step.
int batch_neighbor_build(sgpr_context* h, int64_t N, const BatchGeom& bg, cudaStream_t st, int64_t* n_pairs) {
    h->active_all = true;
    h->n_active = N;
    SGPR_TRY(h->nl_cnt.ensure(sizeof(int) * ((size_t)N * h->S + 1)));
    SGPR_TRY(h->nl_masks.ensure(sizeof(unsigned) * kMaskSlots * ((size_t)N + 1)));
    const Geom unused{};
    SGPR_TRY(launch_count(h, 0, (int)N, unused, nullptr, st, -1, &bg));
    const int nkeys = bg.ncell * h->S;
    const int* rstartT = h->rstart.as<int>() + (nkeys + 1);
    return nl_finish(h, unused, st, rstartT, (int)sizeof(int) * bg.ncell, n_pairs, 0, 0, false, &bg);
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
    SGPR_TRY(launch_count(h, 0, n_own, g, with_halo ? mark : nullptr, st, c0));
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
    SGPR_TRY(launch_count(h, n_own, n_halo, g, nullptr, st, -1));
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
