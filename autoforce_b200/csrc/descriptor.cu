// Per-atom descriptor kernels (SURVEY.md section 8 rows a2-a5, a8).
//
// forward : neighbour displacements -> radial x solid-harmonic expansion c[s,n,lm] ->
//           power spectrum p[s1,s2,n1,n2,l] -> normalised, packed row q_hat
//           (reference: SeSoap.forward / UniversalSoap.forward, descriptor/sesoap.py:161-260,
//            descriptor/soap.py:765-851; Ylm.forward descriptor/ylm.py:113-190;
//            displacements descriptor/atoms.py:365-368).
// backward: g = dE/dq_hat -> dE/dc -> per-neighbour dE/dr_ij -> forces + pair virial
//           (what torch.autograd does in calculator/active.py:587-611; analytic form
//            as in sesoap.py:204-246 and ylm.py:191-222).
//
// One warp per environment.  Forward is two-phase per chunk of 32 neighbours: lanes
// first own one neighbour each (radial + harmonics into shared memory); the chunk is then
// contracted into the expansion coefficients as an FP64 tensor-core micro-GEMM
// (mma.sync.m8n8k4.f64: M = lm, N = (species, n), K = neighbours), and so is the power
// spectrum (per l: c . c^T on the upper-triangle tiles).  Backward stages the next
// environment's rows with cp.async, forms dE/dc as DMMA micro-GEMMs per l, then keeps
// lanes on neighbours; dE/dc lives in shared memory and is broadcast-read.  Both kernels
// have compile-time specialisations for the common descriptor sizes (EXNB / EXACT).
//
// Packed descriptor: the power spectrum is symmetric under (s1,n1)<->(s2,n2)
// (descriptor/sesoap.py:195-203), so only pairs a<=b of a=(s,n) are stored, off-diagonal
// entries scaled by sqrt(2): dot products and norms of packed rows equal those of the
// reference's full [S,S,n,n,L] layout.
#include <algorithm>

#include "sgpr_internal.cuh"

namespace sgpr {

__constant__ HarmCoef c_harm;
__constant__ unsigned char c_l_of_lm[(kMaxL + 1) * (kMaxL + 1)];

int upload_harm_coef() {
    HarmCoef hc;
    fill_harm_coef(hc);
    SGPR_CUDA(cudaMemcpyToSymbol(c_harm, &hc, sizeof(hc)));
    unsigned char l_of[(kMaxL + 1) * (kMaxL + 1)];
    for (int l = 0; l <= kMaxL; ++l)
        for (int k = l * l; k < (l + 1) * (l + 1); ++k) l_of[k] = (unsigned char)l;
    SGPR_CUDA(cudaMemcpyToSymbol(c_l_of_lm, l_of, sizeof(l_of)));
    return SGPR_OK;
}

namespace {

constexpr double kEps = 2.220446049250313e-16;  // torch.finfo(float64).eps, sesoap.py:249

struct EnvSrc {
    // atoms mode
    const AtomRec* atoms;
    const PairRec* pairs;
    const longlong2* nl_rows;   // (begin, end) of each environment's row in pairs
    const int* active;   // env -> cell-order index (nullptr: identity)
    // explicit-environment mode (inducing LCEs)
    const long long* env_first;
    const double* env_r;
    const unsigned char* env_sp;
};

// image-shift cell of a batched step: the lattice vectors of the centre's structure (G = Geom otherwise)
struct CellRef {
    const double* cell;
};

template <bool ENV>
struct Nbr {
    // displacement r_ij (as the reference computes it) and species of neighbour k
    template <class G>
    __device__ static __forceinline__ void load(const EnvSrc& src, const G& g, const AtomRec& ai, long long k,
                                                double& rx, double& ry, double& rz, int& sp, int& j) {
        if (ENV) {
            rx = src.env_r[3 * k];
            ry = src.env_r[3 * k + 1];
            rz = src.env_r[3 * k + 2];
            sp = src.env_sp[k];
            j = -1;
        } else {
            load_pair(src, g, ai, src.pairs[k], rx, ry, rz, sp, j);
        }
    }
    // atoms mode with the pair record already in registers (software-pipelined loops)
    template <class G>
    __device__ static __forceinline__ void load_pair(const EnvSrc& src, const G& g, const AtomRec& ai, const PairRec pr,
                                                     double& rx, double& ry, double& rz, int& sp, int& j) {
        {
            const AtomRec aj = src.atoms[pr.j];
            j = pr.j;
            sp = pr.sp;
            const int i0 = pr.sb[0] - meta_w(aj.meta, 0) + meta_w(ai.meta, 0);
            const int i1 = pr.sb[1] - meta_w(aj.meta, 1) + meta_w(ai.meta, 1);
            const int i2 = pr.sb[2] - meta_w(aj.meta, 2) + meta_w(ai.meta, 2);
            // r = xyz[n] - xyz[a] + (off[...,None]*lll).sum(dim=1)   (descriptor/atoms.py:366-368)
            rx = __dadd_rn(aj.x, -ai.x);
            ry = __dadd_rn(aj.y, -ai.y);
            rz = __dadd_rn(aj.z, -ai.z);
            if ((i0 | i1 | i2) != 0) {   // image shift 0 (the bulk of a large cell): the cell term is an exact + 0.0
                const double S0 = (double)i0, S1 = (double)i1, S2 = (double)i2;
                rx = __dadd_rn(rx, __dadd_rn(__dadd_rn(__dmul_rn(S0, g.cell[0]), __dmul_rn(S1, g.cell[3])), __dmul_rn(S2, g.cell[6])));
                ry = __dadd_rn(ry, __dadd_rn(__dadd_rn(__dmul_rn(S0, g.cell[1]), __dmul_rn(S1, g.cell[4])), __dmul_rn(S2, g.cell[7])));
                rz = __dadd_rn(rz, __dadd_rn(__dadd_rn(__dmul_rn(S0, g.cell[2]), __dmul_rn(S1, g.cell[5])), __dmul_rn(S2, g.cell[8])));
            }
        }
    }
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}

// packed-entry table word: a | b << 8 | l << 16
__device__ __forceinline__ double pspec_entry(const DescParams& dp, const double* c_s, unsigned w, double scale) {
    const int a = w & 0xff, b = (w >> 8) & 0xff, l = (w >> 16) & 0xff;
    const double* ca = c_s + a * dp.L2p + l * l;
    const double* cb = c_s + b * dp.L2p + l * l;
    double s = 0.0;
    for (int k = 0; k < 2 * l + 1; ++k) s += ca[k] * cb[k];
    return s * scale;
}

// ---------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------
// D(8x8) += A(8x4, row) . B(4x8, col) on the FP64 tensor cores.  Fragments: A[lane>>2][lane&3], B[lane&3][lane>>2],
// D[lane>>2][2*(lane&3) + {0,1}].
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// Phase B (expansion coefficients c[s][n][lm] = sum_j f_n(j) Y_lm(j)): one small GEMM per neighbour species on the
// FP64 tensor cores -- M = lm (8-row tiles), N = n (8-column tiles), K = neighbours of the species (4 per step),
// fragments read from the chunk buffer.  (TN, TL only shape the chunk-buffer rows.)
// EXNB > 0: dp.nb == EXNB and dp.lmax == LMAX (bounds, strides and tile predicates fold at compile time)
// BATCH: batched step, image shifts from bcell [B,9] of the centre's structure astr[c]
template <int LMAX, int TN, int TL, bool ENV, int EXNB, bool BATCH = false>
__global__ void __launch_bounds__(128, (LMAX <= 3 ? 7 : 4)) desc_forward_kernel(DescParams dp, Geom g, int n_env, EnvSrc src,
                                                           const int* __restrict__ row_of,
                                                           const unsigned* __restrict__ ptab,
                                                           const double* __restrict__ nnlk, double* __restrict__ phat,
                                                           double* __restrict__ cbuf, double* __restrict__ prow,
                                                           unsigned char* __restrict__ sflag, int per_warp_doubles,
                                                           int stride_, int nbp_, signed char* __restrict__ p8,
                                                           long long p8_slice, int kp1,
                                                           const double* __restrict__ bcell = nullptr,
                                                           const int* __restrict__ astr = nullptr) {
    extern __shared__ __align__(16) double smem[];
    constexpr bool EXACT = EXNB > 0;
    constexpr int kNbp = ((EXNB + TN - 1) / TN) * TN, kL2 = (LMAX + 1) * (LMAX + 1);
    constexpr int kStride = (kNbp + ((kL2 + TL - 1) / TL) * TL) | 1;      // launch_forward's row stride
    const int nbv = EXACT ? EXNB : dp.nb, lmaxv = EXACT ? LMAX : dp.lmax, L2v = EXACT ? kL2 : dp.L2;
    const int L2p = EXACT ? (kL2 | 1) : dp.L2p, nbp = EXACT ? kNbp : nbp_, stride = EXACT ? kStride : stride_;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    double* c_s = smem + (size_t)warp * per_warp_doubles;
    double* buf = c_s + ((dp.csize + 1) & ~1);          // [32][stride]: f[0..nb) | pad | Y[0..L2) | pad
    int* sp_s = reinterpret_cast<int*>(buf + 32 * stride);
    const int g8 = lane >> 2, t4 = lane & 3;   // DMMA fragment coordinates
    const bool all_species = dp.A <= 8 * ((kMaxNB + 7) / 8);
    const int sp_stride = nbv * L2p;  // c[s][n][lm] at (s*nb + n)*L2p + lm
    const int L = lmaxv + 1;
    const int npairs = dp.A * (dp.A + 1) / 2;
    const bool cache_q = dp.D <= 32 * stride;            // packed row fits the (then idle) chunk buffer
    // column (s, n) of this lane's B fragments in the all-species product (loop invariant: no integer division inside)
    constexpr int NT_ = (kMaxNB + 7) / 8;
    int col_s[NT_], col_n[NT_];
#pragma unroll
    for (int nt = 0; nt < NT_; ++nt) {
        const int col = nt * 8 + (lane >> 2);
        col_s[nt] = col / nbv;
        col_n[nt] = col - col_s[nt] * nbv;
    }
    for (int env = blockIdx.x * nwarps + warp; env < n_env; env += gridDim.x * nwarps) {
        long long beg, end;
        AtomRec ai;
        int c = env;
        if (ENV) {
            beg = src.env_first[env];
            end = src.env_first[env + 1];
            ai.x = ai.y = ai.z = 0.0;
            ai.meta = 0;
        } else {
            c = src.active ? src.active[env] : env;
            ai = src.atoms[c];
            const longlong2 row = src.nl_rows[env];
            beg = row.x;
            end = row.y;
        }
        [[maybe_unused]] CellRef cref{nullptr};
        if constexpr (BATCH) cref.cell = bcell + 9 * (size_t)astr[c];
        for (int t = lane; t < dp.csize; t += 32) c_s[t] = 0.0;
        // pass 0: does any neighbour sit (almost) on the z axis?   ylm.py:10-23
        bool hit = false;
        for (long long k = beg + lane; k < end; k += 32) {
            double rx, ry, rz;
            int sp, j;
            if constexpr (BATCH)
                Nbr<ENV>::load(src, cref, ai, k, rx, ry, rz, sp, j);
            else
                Nbr<ENV>::load(src, g, ai, k, rx, ry, rz, sp, j);
            hit |= near_z_axis(rx, ry, rz);   // |x| < a |z| and |y| < a |z| does not depend on the length unit
        }
        const bool flag = __any_sync(0xffffffffu, hit);
        __syncwarp();
        int cur_s = -1;
        constexpr int MT = ((LMAX + 1) * (LMAX + 1) + 7) / 8, NT = (kMaxNB + 7) / 8;
        double acc[MT][NT][2];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
        auto flush = [&](int sp) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const int lm = mt * 8 + g8, n = nt * 8 + 2 * t4;
                    if (lm < L2v) {
                        if (n < nbv) c_s[sp * sp_stride + n * L2p + lm] += acc[mt][nt][0];
                        if (n + 1 < nbv) c_s[sp * sp_stride + (n + 1) * L2p + lm] += acc[mt][nt][1];
                    }
                    acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
                }
        };
        for (long long k0 = beg; k0 < end; k0 += 32) {
            const long long k = k0 + lane;
            if (k < end) {
                double rx, ry, rz;
                int sp, j;
                if constexpr (BATCH)
                    Nbr<ENV>::load(src, cref, ai, k, rx, ry, rz, sp, j);
                else
                    Nbr<ENV>::load(src, g, ai, k, rx, ry, rz, sp, j);
                const double u = dp.radii[sp], ru = dp.rinv[sp];
                const double x = rx * ru, y = ry * ru, z = rz * ru;
                const double d2 = x * x + y * y + z * z;
                const double d = sqrt(d2);
                double R, Rpd;
                radial_fast(d2, d, 1.0, u, dp.rc, dp.rc_inv, R, Rpd);   // R'(d)/d is not needed here
                if (!dp.nbr_enabled[sp]) R = 0.0;   // species outside the descriptor's `b` list
                double* my = buf + lane * stride;
                double fn = R;
                for (int n = 0; n < nbv; ++n) {
                    my[n] = fn;
                    fn *= d2;
                }
                double ys = y, zs = z;
                if (flag) {
                    ys = y - kTinyAngle * z;
                    zs = kTinyAngle * y + z;
                }
                double* yo = my + nbp;
                solid_harmonics<LMAX, false>(c_harm, lmaxv, x, ys, zs,
                                             [&](int idx, double Y, double, double, double) { yo[idx] = Y; });
                sp_s[lane] = sp;
            }
            __syncwarp();
            const int cnt = (int)min((long long)32, end - k0);
            if (all_species) {
                // S*nb <= 8*NT: ONE product for all neighbour species, columns (s, n); B[j][(s, n)] = [s == s_j] f_n(j)
                for (int kk = 0; kk < cnt; kk += 4) {
                    const int jj = kk + t4;
                    const bool ok = jj < cnt;
                    const double* row = buf + jj * stride;
                    const int sj = ok ? sp_s[jj] : -1;
                    double bv[NT];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        bv[nt] = (col_s[nt] == sj) ? row[col_n[nt]] : 0.0;
                    }
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        if (mt * 8 < L2v) {
                            const double av = (ok && mt * 8 + g8 < L2v) ? row[nbp + mt * 8 + g8] : 0.0;
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
                                if (nt * 8 < dp.A) dmma884(acc[mt][nt][0], acc[mt][nt][1], av, bv[nt]);
                        }
                    }
                }
                __syncwarp();
                continue;
            }
            for (int j0 = 0; j0 < cnt;) {
                // run of equal species starting at j0 (atoms: rows are ordered by species; inducing LCEs: any order)
                const int s = sp_s[j0];
                const unsigned diff = __ballot_sync(0xffffffffu, lane > j0 && lane < cnt && sp_s[lane] != s);
                const int j1 = diff ? __ffs(diff) - 1 : cnt;
                if (s != cur_s) {
                    if (cur_s >= 0) flush(cur_s);
                    cur_s = s;
                }
                for (int kk = j0; kk < j1; kk += 4) {
                    const int jj = kk + t4;
                    const bool ok = jj < j1;
                    const double* row = buf + jj * stride;
                    double bv[NT];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) bv[nt] = (ok && nt * 8 + g8 < nbv) ? row[nt * 8 + g8] : 0.0;
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        if (mt * 8 < L2v) {
                            const double av = (ok && mt * 8 + g8 < L2v) ? row[nbp + mt * 8 + g8] : 0.0;
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
                                if (nt * 8 < nbv) dmma884(acc[mt][nt][0], acc[mt][nt][1], av, bv[nt]);
                        }
                    }
                }
                j0 = j1;
            }
            __syncwarp();
        }
        if (all_species) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const int lm = mt * 8 + g8, col = nt * 8 + 2 * t4;   // column (s, n) = row s*nb + n of c
                    if (lm < L2v) {
                        if (col < dp.A) c_s[col * L2p + lm] = acc[mt][nt][0];
                        if (col + 1 < dp.A) c_s[(col + 1) * L2p + lm] = acc[mt][nt][1];
                    }
                }
        } else if (cur_s >= 0) {
            flush(cur_s);
        }
        __syncwarp();
        // power spectrum: lanes over pairs (a <= b), all l of a pair from one pass over c_a, c_b;
        // norm over ALL blocks (sesoap.py:249-251); packed row out
        double ss = 0.0;
        if (cache_q) {
            // p[a, b, l] = sum_m c[a][l m] c[b][l m]: per l a symmetric [A x (2l+1)] . [(2l+1) x A] product on the FP64
            // tensor cores, upper-triangle 8 x 8 tiles only; a lane's two outputs of a tile go to packed entries
            // (tri(a, b), l) -- the same packed order as ptab
            const int AT = (dp.A + 7) >> 3;
            for (int mt = 0; mt < AT; ++mt) {
                const int a = mt * 8 + g8;
                const double* ca = c_s + a * L2p + t4;
                const int tri_a = a * dp.A - ((a * (a - 1)) >> 1) - a;   // tri(a, b) = tri_a + b for b >= a
                for (int nt = mt; nt < AT; ++nt) {
                    const double* cb = c_s + (nt * 8 + g8) * L2p + t4;
                    const int b0 = nt * 8 + 2 * t4;
                    const bool ok0 = a <= b0 && b0 < dp.A, ok1 = a <= b0 + 1 && b0 + 1 < dp.A;
                    const int e0 = (tri_a + b0) * L;
#pragma unroll
                    for (int l = 0; l <= LMAX; ++l) {
                        if (l <= lmaxv) {
                            double d0 = 0.0, d1 = 0.0;
#pragma unroll
                            for (int kk = 0; kk < 2 * l + 1; kk += 4) {
                                // k >= 2l+1 belongs to the next l: zero it in both operands (rows >= A only reach
                                // outputs that are dropped)
                                const bool kok = kk + t4 < 2 * l + 1;
                                const double av = kok ? ca[l * l + kk] : 0.0;
                                const double bv = (nt == mt) ? av : (kok ? cb[l * l + kk] : 0.0);
                                dmma884(d0, d1, av, bv);
                            }
                            if (ok0) {
                                const double q = d0 * nnlk[e0 + l];
                                ss += q * q;
                                buf[e0 + l] = q;
                            }
                            if (ok1) {
                                const double q = d1 * nnlk[e0 + L + l];
                                ss += q * q;
                                buf[e0 + L + l] = q;
                            }
                        }
                    }
                }
            }
        } else {
            for (int pair = lane; pair < npairs; pair += 32) {
                const unsigned w = ptab[pair * L];
                const double* ca = c_s + (w & 0xff) * L2p;
                const double* cb = c_s + ((w >> 8) & 0xff) * L2p;
#pragma unroll
                for (int l = 0; l <= LMAX; ++l) {
                    if (l <= lmaxv) {
                        double sum = 0.0;
#pragma unroll
                        for (int kk = l * l; kk < (l + 1) * (l + 1); ++kk) sum += ca[kk] * cb[kk];
                        const double q = sum * nnlk[pair * L + l];
                        ss += q * q;
                    }
                }
            }
        }
        ss = warp_sum(ss);
        const double P = dp.normalize ? (sqrt(ss) + kEps) : 1.0;
        const double rP = 1.0 / P;
        const size_t row = (size_t)row_of[ENV ? env : c] * dp.ldp;
        __syncwarp();
        if (cache_q) {
            for (int e = lane; e < dp.ldp; e += 32) phat[row + e] = (e < dp.D) ? buf[e] * rP : 0.0;
        } else {
            for (int e = lane; e < dp.ldp; e += 32)
                phat[row + e] = (e < dp.D) ? pspec_entry(dp, c_s, ptab[e], nnlk[e]) * rP : 0.0;
        }
        if (p8) {
            // operand of the tcgen05 kernel-matrix GEMM: 6 balanced base-256 digits of q_hat * 2^46,
            // slice-major, 4 consecutive entries (one 32-bit store per slice) per lane
            // K-chunk-major operand layout of the tcgen05 GEMMs (i8gemm.cu: cm_off): [slice][chunk of 64][row][64]
            const long long prow = (long long)row_of[ENV ? env : c] * 64;
            const long long chunk_stride = p8_slice / kp1 * 64;   // rows per slice * 64
            for (int e4 = lane * 4; e4 < dp.D; e4 += 128) {
                unsigned long long u[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int e = e4 + q;
                    double x = 0.0;
                    if (e < dp.D) x = (cache_q ? buf[e] : pspec_entry(dp, c_s, ptab[e], nnlk[e])) * rP;
                    // bytes of (rint(x 2^46) + bias) ^ bias are the balanced base-256 digits (i8gemm.cu)
                    // rint(x 2^46) via the 1.5 2^52 magic number (|x| <= 1; the 64-bit F2I unit is ~30x slower than a DADD)
                    const long long v = __double_as_longlong(x * 70368744177664.0 + 6755399441055744.0) - 0x4338000000000000ll;
                    u[q] = ((unsigned long long)(v + 0x808080808080ll)) ^ 0x808080808080ull;
                }
                unsigned packed[6];
#pragma unroll
                for (int t = 0; t < 6; ++t) {
                    const int b = 5 - t;   // slice t (most significant first) = byte 5 - t
                    unsigned w0, w1, w2, w3;
                    if (b < 4) {
                        w0 = (unsigned)u[0]; w1 = (unsigned)u[1]; w2 = (unsigned)u[2]; w3 = (unsigned)u[3];
                    } else {
                        w0 = (unsigned)(u[0] >> 32); w1 = (unsigned)(u[1] >> 32); w2 = (unsigned)(u[2] >> 32); w3 = (unsigned)(u[3] >> 32);
                    }
                    const unsigned bb = (unsigned)(b & 3);
                    const unsigned sel = bb | ((4u + bb) << 4);
                    packed[t] = __byte_perm(__byte_perm(w0, w1, sel), __byte_perm(w2, w3, sel), 0x5410);
                }
                const long long off = (long long)(e4 >> 6) * chunk_stride + prow + (e4 & 63);
#pragma unroll
                for (int t = 0; t < 6; ++t) *reinterpret_cast<unsigned*>(p8 + (long long)t * p8_slice + off) = packed[t];
            }
        }
        if (cbuf) {
            for (int t = lane; t < dp.csize; t += 32) cbuf[(size_t)env * dp.csize + t] = c_s[t];
            if (lane == 0) {
                // norm of the row: the backward pass divides by it; for an un-normalised model (P = 1) the covloss
                // needs the self kernel (p.p)^xi instead (calculator/active.py:784-791)
                prow[row_of[c]] = dp.normalize ? P : sqrt(ss);
                sflag[env] = flag ? 1 : 0;
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------
// backward: forces + virial
// ---------------------------------------------------------------------------------
struct BackOut {
    PeerForces peers;            // world > 0: neighbour forces are added into the owner rank's buffer (NVLink)
    double* fcell;               // [N,3] forces in cell order (atomically accumulated)
    double* wpart;               // [gridDim.x, 9] per-block virial partials
    const unsigned char* owned;  // by cell-order index, nullptr = all owned
    const unsigned char* sp_on;  // [S] species has usable inducing points
};

// EXACT: dp.lmax == LMAX and dp.nb == NB (the loop bounds, strides and radial-index predicates fold at compile time)
// BATCH: batched step -- image shifts from bcell [B,9] of the centre's structure astr[c]; each environment writes its
// virial (lane partials, fixed shuffle tree) to wenv [c, 9] instead of the per-block partials
template <int LMAX, int NB, bool EXACT, bool BATCH = false>
__global__ void __launch_bounds__(128, (NB <= 4 ? 4 : 3)) desc_backward_kernel(DescParams dp, Geom g, int n_env, EnvSrc src,
                                                            const int* __restrict__ row_of,
                                                            const double* __restrict__ tvec,
                                                            const double* __restrict__ phat,
                                                            const double* __restrict__ ttab,
                                                            const double* __restrict__ erow,
                                                            const double* __restrict__ prow, double xi,
                                                            const double* __restrict__ cbuf,
                                                            const unsigned char* __restrict__ sflag, BackOut out,
                                                            int per_warp_doubles, const double* __restrict__ bcell = nullptr,
                                                            const int* __restrict__ astr = nullptr,
                                                            double* __restrict__ wenv = nullptr) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double wred[8][9];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    double* T_s = smem + (size_t)warp * per_warp_doubles;   // [D]   dE/dq_hat row, then dE/dq * kappa*nnl * (1 + [a==b])
    double* P_s = T_s + ((dp.D + 1) & ~1);                  // [D]   q_hat row
    double* c_s = P_s + ((dp.D + 1) & ~1);                  // [csize]
    double* D_s = c_s + ((dp.csize + 1) & ~1);              // [csize] dE/dc
    const int L = EXACT ? LMAX + 1 : dp.lmax + 1;
    const int nbv = EXACT ? NB : dp.nb;
    const int L2p = EXACT ? (((LMAX + 1) * (LMAX + 1)) | 1) : dp.L2p;
    const int lmaxv = EXACT ? LMAX : dp.lmax;
    // per-lane operand addresses of the dE/dc micro-GEMM below for A <= 16 (2 row tiles x 4 k-steps): the packed
    // symmetric index tri(a,b) and the row strides do not depend on the environment
    const int g8 = lane >> 2, t4 = lane & 3;
    const bool small_A = dp.A <= 16;
    int toff[2][4], boff[4], doff[2];
    unsigned okm = 0;  // bit ki: b = 4 ki + t4 < A; bit 4 + mi: a = 8 mi + g8 < A
#pragma unroll
    for (int ki = 0; ki < 4; ++ki) {
        const int b = ki * 4 + t4;
        const bool b_ok = b < dp.A;
        okm |= (b_ok ? 1u : 0u) << ki;
        boff[ki] = b_ok ? b * L2p : 0;
#pragma unroll
        for (int mi = 0; mi < 2; ++mi) {
            const int a = mi * 8 + g8;
            const int lo = min(a, b), hi = max(a, b);
            const int tri = lo * dp.A - ((lo * (lo - 1)) >> 1) + (hi - lo);
            toff[mi][ki] = (a < dp.A && b_ok) ? tri * L : 0;   // masked entries read a finite value times bv = 0
        }
    }
#pragma unroll
    for (int mi = 0; mi < 2; ++mi) {
        const int a = mi * 8 + g8;
        okm |= (a < dp.A ? 1u : 0u) << (4 + mi);
        doff[mi] = a * L2p + 2 * t4;
    }
    double Wacc[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) Wacc[q] = 0.0;
    // fused exchange step: which of the peers' two accumulation buffers this step adds into (device-side step parity)
    const long long peer_off = (out.peers.world > 0 && out.peers.parity_src && ((*out.peers.parity_src) & 1)) ? out.peers.parity_stride : 0;

    // The three input rows of an environment (dE/dq_hat, q_hat, expansion coefficients) are only read before the
    // neighbour loop, which is most of an environment's time: the NEXT environment's rows are copied into the same
    // shared-memory buffers asynchronously (cp.async, no register round trip) while that loop runs.
    const int env_stride = gridDim.x * nwarps;
    auto row_of_env = [&](int e) -> int { return e < n_env ? row_of[src.active ? src.active[e] : e] : -1; };
    const bool al16 = ((dp.D | dp.ldp | dp.csize) & 1) == 0;
    auto fetch_rows = [&](int e, int r) {
        const double* tv = tvec + (size_t)r * dp.ldp;
        const double* ph = phat + (size_t)r * dp.ldp;
        const double* cb = cbuf + (size_t)e * dp.csize;
        if (al16) {
            for (int i = 2 * lane; i < dp.D; i += 64) {
                cp_async16(T_s + i, tv + i);
                cp_async16(P_s + i, ph + i);
            }
            for (int i = 2 * lane; i < dp.csize; i += 64) cp_async16(c_s + i, cb + i);
        } else {
            for (int i = lane; i < dp.D; i += 32) {
                cp_async8(T_s + i, tv + i);
                cp_async8(P_s + i, ph + i);
            }
            for (int i = lane; i < dp.csize; i += 32) cp_async8(c_s + i, cb + i);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    {
        const int e0 = blockIdx.x * nwarps + warp, r0 = row_of_env(e0);
        if (r0 >= 0) fetch_rows(e0, r0);
    }
    for (int env = blockIdx.x * nwarps + warp; env < n_env; env += env_stride) {
        const int r_next = row_of_env(env + env_stride);
        const int c = src.active ? src.active[env] : env;
        const AtomRec ai = src.atoms[c];
        const int si = meta_species(ai.meta);
        [[maybe_unused]] CellRef cref{nullptr};
        if constexpr (BATCH) {
            cref.cell = bcell + 9 * (size_t)astr[c];
#pragma unroll
            for (int q = 0; q < 9; ++q) Wacc[q] = 0.0;
        }
        const long long beg = src.nl_rows[env].x, end = src.nl_rows[env].y;
        const bool skip = end == beg || !out.sp_on[si];   // warp-uniform
        const bool flag = sflag[env] != 0;
        // chain rule through the normalisation (sesoap.py:229-235): dE/dq = (g - q_hat (q_hat.g)) / P with
        // q_hat.g = sum_m G_im k_im = xi e_i (the local energy from the kernel-matrix GEMM) -> no dot pass
        const int r = row_of[c];
        // ... times (|p| + eps) / |p| (q_hat = p / (|p| + eps), sesoap.py:249-251): matters only for tiny norms
        const double Pn = dp.normalize ? prow[r] : 1.0;
        const double pg = dp.normalize ? xi * erow[r] * (Pn > 2.0 * kEps ? Pn / (Pn - kEps) : 1.0) : 0.0;
        const double rP = 1.0 / Pn;
        PairRec pr_n;
        pr_n.j = 0;
        const bool have0 = !skip && beg + lane < end;
        if (have0) pr_n = src.pairs[beg + lane];
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();
        if (!skip) {
#pragma unroll 4
            for (int e = lane; e < dp.D; e += 32) T_s[e] = (T_s[e] - P_s[e] * pg) * rP * ttab[e];
        }
        if (have0) asm volatile("prefetch.global.L1 [%0];" ::"l"(src.atoms + pr_n.j));
        __syncwarp();
        // dE/dc[a][lm] = sum_b T[tri(a,b), l] c[b][lm],  tri(a,b) = rs(min) + |a-b|, rs(x) = x A - x(x-1)/2
        // = per l one symmetric [A x A] . [A x (2l+1)] product on the FP64 tensor cores (M = a, N = m, K = b)
        if (skip) {
        } else if (small_A) {
#pragma unroll
            for (int l = 0; l <= LMAX; ++l) {
                if (l > lmaxv) break;
                const int nm = 2 * l + 1, lm0 = l * l;
#pragma unroll
                for (int nn0 = 0; nn0 < nm; nn0 += 8) {
                    // columns n >= nm and rows a >= A of the product are never stored; k-entries b >= A are zeroed.
                    // Columns n >= nm are not read either: past the last l of row b = A-1 they lie beyond the c block,
                    // and for lmax = 0 with A < 5 beyond this warp's shared-memory slice (for the last warp: past the
                    // end of the block's allocation)
                    const double* cl = c_s + lm0 + nn0 + g8;
                    const bool n_ok = nn0 + g8 < nm;
                    double bv[4];
#pragma unroll
                    for (int ki = 0; ki < 4; ++ki) bv[ki] = (n_ok && ((okm >> ki) & 1u)) ? cl[boff[ki]] : 0.0;
#pragma unroll
                    for (int mi = 0; mi < 2; ++mi) {
                        if (mi * 8 < dp.A) {
                            double d0 = 0.0, d1 = 0.0;
#pragma unroll
                            for (int ki = 0; ki < 4; ++ki)
                                if (ki * 4 < dp.A) dmma884(d0, d1, T_s[toff[mi][ki] + l], bv[ki]);
                            const int n = nn0 + 2 * t4;
                            if ((okm >> (4 + mi)) & 1u) {
                                if (n < nm) D_s[doff[mi] + lm0 + nn0] = d0;
                                if (n + 1 < nm) D_s[doff[mi] + lm0 + nn0 + 1] = d1;
                            }
                        }
                    }
                }
            }
        } else {
            for (int l = 0; l < L; ++l) {
                const int nm = 2 * l + 1, lm0 = l * l;
                for (int nn0 = 0; nn0 < nm; nn0 += 8) {
                    const bool nB_ok = nn0 + g8 < nm;
                    const double* cl = c_s + lm0 + nn0 + g8;
                    for (int m0 = 0; m0 < dp.A; m0 += 8) {
                        const int a = m0 + g8;
                        const bool a_ok = a < dp.A;
                        double d0 = 0.0, d1 = 0.0;
                        for (int kk = 0; kk < dp.A; kk += 4) {
                            const int b = kk + t4;
                            const bool b_ok = b < dp.A;
                            const int lo = min(a, b), hi = max(a, b);
                            const int tri = lo * dp.A - ((lo * (lo - 1)) >> 1) + (hi - lo);
                            const double av = (a_ok && b_ok) ? T_s[tri * L + l] : 0.0;
                            const double bv = (nB_ok && b_ok) ? cl[b * L2p] : 0.0;
                            dmma884(d0, d1, av, bv);
                        }
                        const int n = nn0 + 2 * t4;
                        if (a_ok) {
                            if (n < nm) D_s[a * L2p + lm0 + n] = d0;
                            if (n + 1 < nm) D_s[a * L2p + lm0 + n + 1] = d1;
                        }
                    }
                }
            }
        }
        __syncwarp();
        if (r_next >= 0) fetch_rows(env + env_stride, r_next);
        if (skip) continue;
        double Fx = 0.0, Fy = 0.0, Fz = 0.0;
        const bool own_i = out.owned ? (out.owned[c] != 0) : true;
        for (long long k = beg + lane; k < end; k += 32) {
            double rx, ry, rz;
            int sp, j;
            // the pair record of this pass was fetched one pass ahead and its atom record prefetched: the dependent
            // pairs -> atoms gather is otherwise two exposed L2 round trips per pass
            const PairRec pr = pr_n;
            const bool more = k + 32 < end;
            if (more) pr_n = src.pairs[k + 32];
            if constexpr (BATCH)
                Nbr<false>::load_pair(src, cref, ai, pr, rx, ry, rz, sp, j);
            else
                Nbr<false>::load_pair(src, g, ai, pr, rx, ry, rz, sp, j);
            const double u = dp.radii[sp], ru = dp.rinv[sp];
            const double x = rx * ru, y = ry * ru, z = rz * ru;
            const double d2 = x * x + y * y + z * z;
            const double rd = rsqrt(d2);
            const double d = d2 * rd;
            double R, Rpd;
            radial_fast(d2, d, rd, u, dp.rc, dp.rc_inv, R, Rpd);
            if (!dp.nbr_enabled[sp]) {
                R = 0.0;
                Rpd = 0.0;
            }
            if (more) asm volatile("prefetch.global.L1 [%0];" ::"l"(src.atoms + pr_n.j));
            double f[NB], hh[NB], Tn[NB];
            {
                double pw = 1.0;  // d2^(n-1)
                f[0] = R;
                hh[0] = Rpd;
                Tn[0] = 0.0;
#pragma unroll
                for (int n = 1; n < NB; ++n) {
                    f[n] = f[n - 1] * d2;
                    hh[n] = Rpd * (pw * d2) + 2.0 * n * R * pw;
                    pw *= d2;
                    Tn[n] = 0.0;
                }
            }
            double ys = y, zs = z;
            if (flag) {
                ys = y - kTinyAngle * z;
                zs = kTinyAngle * y + z;
            }
            const double* Dj = D_s + sp * nbv * L2p;
            double gx = 0.0, gy = 0.0, gz = 0.0;
            solid_harmonics<LMAX, true>(c_harm, lmaxv, x, ys, zs,
                                        [&](int idx, double Y, double dYx, double dYy, double dYz) {
                                            double B = 0.0;
#pragma unroll
                                            for (int n = 0; n < NB; ++n) {
                                                if (n < nbv) {
                                                    const double dc = Dj[n * L2p + idx];
                                                    B += dc * f[n];
                                                    Tn[n] += dc * Y;
                                                }
                                            }
                                            gx += B * dYx;
                                            gy += B * dYy;
                                            gz += B * dYz;
                                        });
            if (flag) {  // transpose of the shear, ylm.py:212-220
                const double t = gy;
                gy = t + kTinyAngle * gz;
                gz = -kTinyAngle * t + gz;
            }
            double rad = 0.0;
#pragma unroll
            for (int n = 0; n < NB; ++n)
                if (n < nbv) rad += Tn[n] * hh[n];
            const double Gx = (rad * x + gx) * ru, Gy = (rad * y + gy) * ru, Gz = (rad * z + gz) * ru;
            if (own_i) {
                Fx += Gx;
                Fy += Gy;
                Fz += Gz;
                Wacc[0] += rx * Gx; Wacc[1] += rx * Gy; Wacc[2] += rx * Gz;
                Wacc[3] += ry * Gx; Wacc[4] += ry * Gy; Wacc[5] += ry * Gz;
                Wacc[6] += rz * Gx; Wacc[7] += rz * Gy; Wacc[8] += rz * Gz;
            }
            if (out.peers.world > 0) {
                // atom-sharded: everything is accumulated in THIS rank's buffer (indexed by the global cell order); the
                // entries of atoms other ranks own are pushed to their owners afterwards, one remote add per atom and
                // component instead of one per pair (p2p_push_kernel, api.cu)
                double* dst = out.fcell + peer_off + 3 * (size_t)j;
                atomicAdd(dst, -Gx);
                atomicAdd(dst + 1, -Gy);
                atomicAdd(dst + 2, -Gz);
            } else if (!out.owned || out.owned[j]) {
                atomicAdd(out.fcell + 3 * (size_t)j, -Gx);
                atomicAdd(out.fcell + 3 * (size_t)j + 1, -Gy);
                atomicAdd(out.fcell + 3 * (size_t)j + 2, -Gz);
            }
        }
        Fx = warp_sum(Fx);
        Fy = warp_sum(Fy);
        Fz = warp_sum(Fz);
        if (lane == 0 && own_i) {
            double* fown = out.fcell + peer_off;
            atomicAdd(fown + 3 * (size_t)c, Fx);
            atomicAdd(fown + 3 * (size_t)c + 1, Fy);
            atomicAdd(fown + 3 * (size_t)c + 2, Fz);
        }
        if constexpr (BATCH) {
#pragma unroll
            for (int q = 0; q < 9; ++q) Wacc[q] = warp_sum(Wacc[q]);
            if (lane == 0)
#pragma unroll
                for (int q = 0; q < 9; ++q) wenv[9 * (size_t)c + q] = Wacc[q];
        }
        __syncwarp();
    }
    if constexpr (!BATCH) {
#pragma unroll
        for (int q = 0; q < 9; ++q) Wacc[q] = warp_sum(Wacc[q]);
        if (lane == 0)
#pragma unroll
            for (int q = 0; q < 9; ++q) wred[warp][q] = Wacc[q];
        __syncthreads();
        if (threadIdx.x < 9) {
            double s = 0.0;
            for (int w = 0; w < nwarps; ++w) s += wred[w][threadIdx.x];
            out.wpart[blockIdx.x * 9 + threadIdx.x] = s;
        }
    }
}

// ---------------------------------------------------------------------------------
// training-time kernels: d Ke[m] / d x for a tile of inducing LCEs at once
// ---------------------------------------------------------------------------------
// Per environment i (centre species s) and inducing LCE m of species s, with the cotangent of the backward pass above
// seeded by column m (g = xi k^(xi-1) z_hat_m, e = k^xi):
//   T_m[e]     = (xi k^(xi-1) z_m[e] - q_i[e] pg) / P * ttab[e]              (desc_backward_kernel's T)
//   dKe/dc[a,lm] = sum_b T_m[tri(a,b), l] c[b,lm] = alpha_m U_m[a,lm] - beta_m V[a,lm]
//   U_m = sum_b (z_m ttab)[tri(a,b), l] c[b,lm],  V = sum_b (q_i ttab)[tri(a,b), l] c[b,lm]  (m-independent)
// and every pair contracts its d c / d r_ij block (radial x harmonic gradients, computed once per pair) against the
// dKe/dc rows of all LCEs of the tile.  One block per (environment, tile of MT = warps x MM LCEs); warp w owns LCEs
// w*MM .. w*MM+MM-1 of the tile and each lane one pair of a chunk of 32.
struct JacArgs {
    const int* sel;          // [n_sel] sorted inducing positions evaluated, grouped by central species
    const int* sel_col;      // [n_sel] output column of each
    int sel_first[kMaxSpecies + 1];
    int n_tiles;             // blocks per environment
    int ncol;                // columns of J and W
    long long n_atoms;       // rows of J
    double* J;               // [ncol, n_atoms, 3], caller's atom order (accumulated)
    double* W;               // [B, ncol, 9] (accumulated)
    const double* cells;     // [B, 9] lattice vectors of the image shifts
    const int* astr;         // [N] structure of a cell-order atom (nullptr: one structure)
};

struct JacLayout {
    int off_V, off_D, off_R;   // doubles from the start of shared memory
    int prs;                   // stride of a pair record (doubles, odd)
    int o_Y, o_xyz;            // offsets inside a pair record: f[nb] hh[nb] Y[L2] dYx[L2] dYy[L2] dYz[L2] x y z ru rx ry rz
    int dpad;                  // per-warp T_m staging stride; 0: T_m is read from global memory
};

// out[a*L2p + lm] = sum_b T[tri(a,b), l] c[b, lm] for o = a*L2 + lm in [o0, A*L2) step ostep; T from shared memory (Ts)
// or as zg[e] * ttab[e]
template <class Store>
__device__ __forceinline__ void jac_contract(const DescParams& dp, int L, int L2, int L2p, const double* Ts,
                                             const double* __restrict__ zg, const double* __restrict__ ttab,
                                             const double* c_s, int o0, int ostep, Store&& store) {
    const int A = dp.A;
    for (int o = o0; o < A * L2; o += ostep) {
        const int a = o / L2, lm = o - a * L2, l = c_l_of_lm[lm];
        const int rs_a = a * A - ((a * (a - 1)) >> 1);
        int rs_b = 0;   // rs(b) = b A - b (b-1) / 2
        double s = 0.0;
        for (int b = 0; b < A; ++b) {
            const int e = (b < a ? rs_b + (a - b) : rs_a + (b - a)) * L + l;
            const double t = Ts ? Ts[e] : zg[e] * ttab[e];
            s = fma(t, c_s[b * L2p + lm], s);
            rs_b += A - b;
        }
        store(a * L2p + lm, s);
    }
}

template <int LMAX, int NB, bool EXACT, int MM>
__global__ void __launch_bounds__(128, 1) jacobian_kernel(DescParams dp, EnvSrc src, JacLayout lay, JacArgs out,
                                                          const int* __restrict__ row_of, const double* __restrict__ phat,
                                                          const double* __restrict__ ttab, const double* __restrict__ prow,
                                                          const double* __restrict__ zhat, double xi, int xi_int,
                                                          const double* __restrict__ cbuf,
                                                          const unsigned char* __restrict__ sflag) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5, MT = nw * MM;
    const int env = blockIdx.x / out.n_tiles, tile = blockIdx.x - env * out.n_tiles;
    const int c = src.active ? src.active[env] : env;
    const AtomRec ai = src.atoms[c];
    const int si = meta_species(ai.meta);
    const long long beg = src.nl_rows[env].x, end = src.nl_rows[env].y;
    const int t0 = out.sel_first[si] + tile * MT, t1 = out.sel_first[si + 1];
    // lone centres (constant K), excluded centres (K = 0) and tiles past the species' LCEs: nothing to add
    if (t0 >= t1 || end == beg || !dp.central_enabled[si]) return;
    const int L = EXACT ? LMAX + 1 : dp.lmax + 1;
    const int nbv = EXACT ? NB : dp.nb;
    const int L2v = EXACT ? (LMAX + 1) * (LMAX + 1) : dp.L2;
    const int L2p = EXACT ? (((LMAX + 1) * (LMAX + 1)) | 1) : dp.L2p;
    const int lmaxv = EXACT ? LMAX : dp.lmax;
    double* c_s = smem;
    double* V_s = smem + lay.off_V;
    double* Dt = smem + lay.off_D;   // [MT][csize] dKe/dc of the tile's LCEs
    double* R = smem + lay.off_R;    // T_m staging, then pair records
    const int r = row_of[c];
    const double* q = phat + (size_t)r * dp.ldp;
    for (int t = threadIdx.x; t < dp.csize; t += blockDim.x) c_s[t] = cbuf[(size_t)env * dp.csize + t];
    if (lay.dpad)
        for (int e = threadIdx.x; e < dp.D; e += blockDim.x) R[e] = q[e] * ttab[e];
    __syncthreads();
    jac_contract(dp, L, L2v, L2p, lay.dpad ? R : nullptr, q, ttab, c_s, threadIdx.x, blockDim.x,
                 [&](int o, double s) { V_s[o] = s; });
    __syncthreads();
    // chain rule through the normalisation as desc_backward_kernel applies it
    const double Pn = dp.normalize ? prow[r] : 1.0;
    const double rP = 1.0 / Pn;
    const double nfac = (Pn > 2.0 * kEps ? Pn / (Pn - kEps) : 1.0);
    double* Tw = lay.dpad ? R + (size_t)warp * lay.dpad : nullptr;
#pragma unroll 1
    for (int mm = 0; mm < MM; ++mm) {
        const int t = t0 + warp * MM + mm;
        if (t >= t1) break;   // warp-uniform
        const double* z = zhat + (size_t)out.sel[t] * dp.ldp;
        double k = 0.0;
        for (int e = lane; e < dp.D; e += 32) {
            const double zv = z[e];
            k = fma(q[e], zv, k);
            if (Tw) Tw[e] = zv * ttab[e];
        }
        k = warp_sum(k);
        double pw = 1.0;
        if (xi_int >= 1) {
            for (int u = 1; u < xi_int; ++u) pw *= k;
        } else {
            pw = pow(k, xi - 1.0);
        }
        const double cm = xi * pw, em = pw * k;
        const double pg = dp.normalize ? xi * em * nfac : 0.0;
        const double alpha = cm * rP, beta = pg * rP;
        double* Dm = Dt + (size_t)(warp * MM + mm) * dp.csize;
        __syncwarp();
        jac_contract(dp, L, L2v, L2p, Tw, z, ttab, c_s, lane, 32,
                     [&](int o, double s) { Dm[o] = alpha * s - beta * V_s[o]; });
        __syncwarp();
    }
    __syncthreads();   // R becomes the pair-record buffer

    const int b = out.astr ? out.astr[c] : 0;
    const CellRef cref{out.cells + 9 * (size_t)b};
    const bool flag = sflag[env] != 0;
    int* pint = reinterpret_cast<int*>(R + 32 * lay.prs);   // [32] species, [32] caller's index of j
    bool ok[MM];
    int col[MM];
#pragma unroll
    for (int mm = 0; mm < MM; ++mm) {
        const int t = t0 + warp * MM + mm;
        ok[mm] = t < t1;
        col[mm] = ok[mm] ? out.sel_col[t] : 0;
    }
    double Gi[MM][3], Wa[MM][9];
#pragma unroll
    for (int mm = 0; mm < MM; ++mm) {
#pragma unroll
        for (int q3 = 0; q3 < 3; ++q3) Gi[mm][q3] = 0.0;
#pragma unroll
        for (int q9 = 0; q9 < 9; ++q9) Wa[mm][q9] = 0.0;
    }
    for (long long k0 = beg; k0 < end; k0 += 32) {
        if (warp == 0) {
            const long long k = k0 + lane;
            double* my = R + (size_t)lane * lay.prs;
            if (k < end) {
                double rx, ry, rz;
                int sp, j;
                Nbr<false>::load_pair(src, cref, ai, src.pairs[k], rx, ry, rz, sp, j);
                const double u = dp.radii[sp], ru = dp.rinv[sp];
                const double x = rx * ru, y = ry * ru, z = rz * ru;
                const double d2 = x * x + y * y + z * z;
                const double rd = rsqrt(d2);
                const double d = d2 * rd;
                double Rr, Rpd;
                radial_fast(d2, d, rd, u, dp.rc, dp.rc_inv, Rr, Rpd);
                if (!dp.nbr_enabled[sp]) {
                    Rr = 0.0;
                    Rpd = 0.0;
                }
                double pw = 1.0;  // d2^(n-1)
                my[0] = Rr;
                my[nbv] = Rpd;
                double fn = Rr;
                for (int n = 1; n < nbv; ++n) {
                    fn *= d2;
                    my[n] = fn;
                    my[nbv + n] = Rpd * (pw * d2) + 2.0 * n * Rr * pw;
                    pw *= d2;
                }
                double ys = y, zs = z;
                if (flag) {
                    ys = y - kTinyAngle * z;
                    zs = kTinyAngle * y + z;
                }
                double* yo = my + lay.o_Y;
                solid_harmonics<LMAX, true>(c_harm, lmaxv, x, ys, zs,
                                            [&](int idx, double Y, double dYx, double dYy, double dYz) {
                                                yo[idx] = Y;
                                                yo[L2v + idx] = dYx;
                                                if (flag) {  // transpose of the shear, ylm.py:212-220 (linear: per component)
                                                    yo[2 * L2v + idx] = dYy + kTinyAngle * dYz;
                                                    yo[3 * L2v + idx] = -kTinyAngle * dYy + dYz;
                                                } else {
                                                    yo[2 * L2v + idx] = dYy;
                                                    yo[3 * L2v + idx] = dYz;
                                                }
                                            });
                double* xyz = my + lay.o_xyz;
                xyz[0] = x; xyz[1] = y; xyz[2] = z; xyz[3] = ru;
                xyz[4] = rx; xyz[5] = ry; xyz[6] = rz;
                pint[lane] = sp;
                pint[32 + lane] = meta_orig(src.atoms[j].meta);
            }
        }
        __syncthreads();
        const int cnt = (int)min((long long)32, end - k0);
        if (lane < cnt) {
            const double* my = R + (size_t)lane * lay.prs;
            const int sp = pint[lane];
            const long long jo = pint[32 + lane];
            double f[NB], hh[NB];
#pragma unroll
            for (int n = 0; n < NB; ++n) {
                f[n] = n < nbv ? my[n] : 0.0;
                hh[n] = n < nbv ? my[nbv + n] : 0.0;
            }
            double Tn[MM][NB], gx[MM], gy[MM], gz[MM];
            const double* Db[MM];
#pragma unroll
            for (int mm = 0; mm < MM; ++mm) {
                gx[mm] = gy[mm] = gz[mm] = 0.0;
#pragma unroll
                for (int n = 0; n < NB; ++n) Tn[mm][n] = 0.0;
                Db[mm] = Dt + (size_t)(warp * MM + mm) * dp.csize + sp * nbv * L2p;
            }
            const double* yo = my + lay.o_Y;
#pragma unroll 2
            for (int lm = 0; lm < L2v; ++lm) {
                const double Y = yo[lm], dx = yo[L2v + lm], dy = yo[2 * L2v + lm], dz = yo[3 * L2v + lm];
#pragma unroll
                for (int mm = 0; mm < MM; ++mm) {
                    double B = 0.0;
#pragma unroll
                    for (int n = 0; n < NB; ++n) {
                        if (n < nbv) {
                            const double dc = Db[mm][n * L2p + lm];
                            B = fma(dc, f[n], B);
                            Tn[mm][n] = fma(dc, Y, Tn[mm][n]);
                        }
                    }
                    gx[mm] = fma(B, dx, gx[mm]);
                    gy[mm] = fma(B, dy, gy[mm]);
                    gz[mm] = fma(B, dz, gz[mm]);
                }
            }
            const double* xyz = my + lay.o_xyz;
            const double x = xyz[0], y = xyz[1], z = xyz[2], ru = xyz[3], rx = xyz[4], ry = xyz[5], rz = xyz[6];
#pragma unroll
            for (int mm = 0; mm < MM; ++mm) {
                if (!ok[mm]) continue;
                double rad = 0.0;
#pragma unroll
                for (int n = 0; n < NB; ++n)
                    if (n < nbv) rad += Tn[mm][n] * hh[n];
                const double Gx = (rad * x + gx[mm]) * ru, Gy = (rad * y + gy[mm]) * ru, Gz = (rad * z + gz[mm]) * ru;
                double* Jj = out.J + ((size_t)col[mm] * out.n_atoms + jo) * 3;
                atomicAdd(Jj, Gx);
                atomicAdd(Jj + 1, Gy);
                atomicAdd(Jj + 2, Gz);
                Gi[mm][0] -= Gx; Gi[mm][1] -= Gy; Gi[mm][2] -= Gz;
                Wa[mm][0] += rx * Gx; Wa[mm][1] += rx * Gy; Wa[mm][2] += rx * Gz;
                Wa[mm][3] += ry * Gx; Wa[mm][4] += ry * Gy; Wa[mm][5] += ry * Gz;
                Wa[mm][6] += rz * Gx; Wa[mm][7] += rz * Gy; Wa[mm][8] += rz * Gz;
            }
        }
        __syncthreads();
    }
    const long long io = meta_orig(ai.meta);
#pragma unroll
    for (int mm = 0; mm < MM; ++mm) {
        if (!ok[mm]) continue;   // warp-uniform
#pragma unroll
        for (int q3 = 0; q3 < 3; ++q3) Gi[mm][q3] = warp_sum(Gi[mm][q3]);
#pragma unroll
        for (int q9 = 0; q9 < 9; ++q9) Wa[mm][q9] = warp_sum(Wa[mm][q9]);
        if (lane == 0) {
            double* Ji = out.J + ((size_t)col[mm] * out.n_atoms + io) * 3;
#pragma unroll
            for (int q3 = 0; q3 < 3; ++q3) atomicAdd(Ji + q3, Gi[mm][q3]);
            double* Wb = out.W + ((size_t)b * out.ncol + col[mm]) * 9;
#pragma unroll
            for (int q9 = 0; q9 < 9; ++q9) atomicAdd(Wb + q9, Wa[mm][q9]);
        }
    }
}

// packed row -> the reference's dense block layout [S,S,nb,nb,L]
__global__ void unpack_kernel(DescParams dp, long long rows, const double* __restrict__ packed,
                              const int* __restrict__ src_row, double* __restrict__ full) {
    const int L = dp.lmax + 1;
    const long long dfull = (long long)dp.A * dp.A * L;
    const long long total = rows * dfull;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long r = t / dfull;
        int o = (int)(t - r * dfull);
        const int l = o % L; o /= L;
        const int n2 = o % dp.nb; o /= dp.nb;
        const int n1 = o % dp.nb; o /= dp.nb;
        const int s2 = o % dp.S;
        const int s1 = o / dp.S;
        const int a = s1 * dp.nb + n1, b = s2 * dp.nb + n2;
        const int lo = min(a, b), hi = max(a, b);
        const int tri = lo * dp.A - (lo * (lo - 1)) / 2 + (hi - lo);
        const double v = packed[(size_t)(src_row ? src_row[r] : r) * dp.ldp + tri * L + l];
        full[t] = (a == b) ? v : v * 0.70710678118654752440;
    }
}

struct Launch {
    int warps;
    size_t smem;
    int per_warp;
};

Launch plan_forward(const DescParams& dp, int stride) {
    // c block + 32 neighbour rows + 32 species ints
    int per_warp = ((dp.csize + 1) & ~1) + 32 * stride + 16;
    int warps = 4;
    while (warps > 1 && (size_t)warps * per_warp * 8 > 200 * 1024) warps >>= 1;
    return {warps, (size_t)warps * per_warp * 8, per_warp};
}
Launch plan_backward(const DescParams& dp) {
    int per_warp = 2 * ((dp.D + 1) & ~1) + 2 * ((dp.csize + 1) & ~1);
    int warps = 4;
    while (warps > 1 && (size_t)warps * per_warp * 8 > 200 * 1024) warps >>= 1;
    return {warps, (size_t)warps * per_warp * 8, per_warp};
}

template <int LMAX, int TN, int TL, bool ENV, int EXNB, bool BATCH>
int launch_forward(sgpr_context* h, const Geom& g, int n_env, const EnvSrc& src, const int* row_of, double* phat,
                   double* cbuf, double* pnorm, unsigned char* sflag, cudaStream_t st, const BatchGeom* bg) {
    const DescParams& dp = h->dp;
    // row of a neighbour in the chunk buffer: f padded to whole n tiles, Y padded to whole lm tiles
    const int nbp = ((dp.nb + TN - 1) / TN) * TN;
    int stride = nbp + ((dp.L2 + TL - 1) / TL) * TL;
    if ((stride & 1) == 0) stride += 1;  // odd stride: lanes writing their own row hit distinct banks
    if (((dp.L2 + TL - 1) / TL) * ((dp.nb + TN - 1) / TN) > 32) {
        set_error("internal: forward tile shape does not cover the components");
        return SGPR_ERR_INVALID;
    }
    Launch L = plan_forward(dp, stride);
    if ((size_t)L.per_warp * 8 > 200 * 1024) {
        set_error("descriptor too large for shared memory (S=%d nmax=%d lmax=%d)", dp.S, dp.nb - 1, dp.lmax);
        return SGPR_ERR_INVALID;
    }
    auto kern = desc_forward_kernel<LMAX, TN, TL, ENV, EXNB, BATCH>;
    SGPR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
    int grid = (n_env + L.warps - 1) / L.warps;
    // one resident wave: environments are dealt round-robin to warps, so a grid that is not a whole number of waves
    // leaves the machine partly idle for the whole last wave
    static thread_local size_t occ_smem = ~(size_t)0;
    static thread_local int occ_blocks = 0;
    if (occ_smem != L.smem) {
        int nb = 0;
        SGPR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, L.warps * 32, L.smem));
        occ_blocks = nb > 0 ? nb : 1;
        occ_smem = L.smem;
    }
    const int maxgrid = h->sm_count * occ_blocks;
    if (grid > maxgrid) grid = maxgrid;
    if (grid < 1) grid = 1;
    kern<<<grid, L.warps * 32, L.smem, st>>>(dp, g, n_env, src, row_of, h->ptab.as<unsigned>(), h->nnlk.as<double>(), phat,
                                             cbuf, pnorm, sflag, L.per_warp, stride, nbp,
                                             (!ENV && h->use_i8_now) ? h->p8.as<signed char>() : nullptr,
                                             (long long)h->i8_cap_rows * h->i8_kp1, h->i8_kp1, bg ? bg->cells : nullptr,
                                             bg ? bg->astr : nullptr);
    SGPR_CUDA(cudaGetLastError());
    h->stats.kernel_launches += 1;
    return SGPR_OK;
}

template <bool ENV, bool BATCH = false>
int dispatch_forward(sgpr_context* h, const Geom& g, int n_env, const EnvSrc& src, const int* row_of, double* phat,
                     double* cbuf, double* pnorm, unsigned char* sflag, cudaStream_t st, const BatchGeom* bg = nullptr) {
    const int lmax = h->dp.lmax, nb = h->dp.nb;
    // (LMAX bucket, n-tile, lm-tile): ceil(L2/TL) * ceil(nb/TN) <= 32 lanes
#define FWD(LM, TN, TL) return launch_forward<LM, TN, TL, ENV, 0, BATCH>(h, g, n_env, src, row_of, phat, cbuf, pnorm, sflag, st, bg)
    if (lmax == 3 && nb == 4)   // the reference's default descriptor
        return launch_forward<3, 2, 1, ENV, 4, BATCH>(h, g, n_env, src, row_of, phat, cbuf, pnorm, sflag, st, bg);
    if (lmax <= 3 && nb <= 4) FWD(3, 2, 1);
    if (lmax == 6 && nb == 9)   // the high-resolution configuration (lmax 6, nmax 8)
        return launch_forward<6, 3, 5, ENV, 9, BATCH>(h, g, n_env, src, row_of, phat, cbuf, pnorm, sflag, st, bg);
    if (lmax <= 3 && nb <= 8) FWD(3, 4, 1);
    if (lmax <= 3) FWD(3, 6, 1);
    if (lmax <= 6 && nb <= 6) FWD(6, 2, 5);
    if (lmax <= 6 && nb <= 9) FWD(6, 3, 5);
    if (lmax <= 6) FWD(6, 4, 5);
    if (lmax <= 8) FWD(8, 6, 6);
#undef FWD
    set_error("unsupported descriptor size lmax=%d nmax=%d", lmax, h->dp.nb - 1);
    return SGPR_ERR_INVALID;
}

template <int LMAX, int NB, bool EXACT, bool BATCH>
int launch_backward(sgpr_context* h, const Geom& g, int n_env, const EnvSrc& src, const BackOut& out, int grid,
                    cudaStream_t st, const BatchGeom* bg) {
    const DescParams& dp = h->dp;
    Launch L = plan_backward(dp);
    if ((size_t)L.per_warp * 8 > 200 * 1024) {
        set_error("descriptor too large for shared memory (S=%d nmax=%d lmax=%d)", dp.S, dp.nb - 1, dp.lmax);
        return SGPR_ERR_INVALID;
    }
    auto kern = desc_backward_kernel<LMAX, NB, EXACT, BATCH>;
    SGPR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
    kern<<<grid, L.warps * 32, L.smem, st>>>(dp, g, n_env, src, h->rowof.as<int>() + (h->last_N + 1),
                                             h->gvec.as<double>(), h->phat.as<double>(), h->ttab.as<double>(),
                                             h->erow.as<double>(), h->prow.as<double>(), h->xi, h->cbuf.as<double>(),
                                             h->sflag.as<unsigned char>(), out, L.per_warp, bg ? bg->cells : nullptr,
                                             bg ? bg->astr : nullptr, bg ? h->wenv.as<double>() : nullptr);
    SGPR_CUDA(cudaGetLastError());
    h->stats.kernel_launches += 1;
    return SGPR_OK;
}

// shared memory of the Jacobian kernel: warps per block, layout and bytes (false: not even one warp fits)
bool plan_jacobian(const DescParams& dp, int MM, JacLayout& lay, int& nw, size_t& smem) {
    lay = JacLayout{};
    lay.o_Y = 2 * dp.nb;
    lay.o_xyz = lay.o_Y + 4 * dp.L2;
    lay.prs = (lay.o_xyz + 7) | 1;
    const int pair_doubles = 32 * lay.prs + 32;   // records + 64 ints
    const size_t cap = 220 * 1024;
    for (nw = 4;; nw >>= 1) {
        const int mt = nw * MM;
        const int dpad = (dp.D + 1) & ~1;
        const size_t fixed = (size_t)(2 + mt) * ((dp.csize + 1) & ~1);
        lay.dpad = dpad;
        size_t rsz = std::max<size_t>((size_t)nw * dpad, pair_doubles);
        if ((fixed + rsz) * 8 > cap) {   // read T_m from global memory instead of staging it
            lay.dpad = 0;
            rsz = pair_doubles;
        }
        smem = (fixed + rsz) * 8;
        if (smem <= cap) return true;
        if (nw == 1) return false;
    }
}

template <int LMAX, int NB, bool EXACT>
int launch_jacobian(sgpr_context* h, const EnvSrc& src, const JacArgs& a, int max_sel, cudaStream_t st) {
    constexpr int MM = NB <= 4 ? 4 : 2;   // LCEs per warp: the register tile of the pair contraction
    const DescParams& dp = h->dp;
    const int na = (int)h->n_active;
    JacLayout lay;
    int nw;
    size_t smem;
    if (!plan_jacobian(dp, MM, lay, nw, smem)) {
        set_error("descriptor too large for the Jacobian kernel (S=%d nmax=%d lmax=%d)", dp.S, dp.nb - 1, dp.lmax);
        return SGPR_ERR_INVALID;
    }
    const int csp = (dp.csize + 1) & ~1;
    lay.off_V = csp;
    lay.off_D = 2 * csp;
    lay.off_R = (2 + nw * MM) * csp;
    JacArgs args = a;
    args.n_tiles = (max_sel + nw * MM - 1) / (nw * MM);
    const long long grid = (long long)na * args.n_tiles;
    if (grid == 0) return SGPR_OK;
    if (grid > 0x7fffffffll) {
        set_error("too many environments x inducing tiles for one Jacobian launch (%lld)", grid);
        return SGPR_ERR_INVALID;
    }
    auto kern = jacobian_kernel<LMAX, NB, EXACT, MM>;
    SGPR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)grid, nw * 32, smem, st>>>(dp, src, lay, args, h->rowof.as<int>() + (h->last_N + 1), h->phat.as<double>(),
                                               h->ttab.as<double>(), h->prow.as<double>(), h->zhat.as<double>(), h->xi,
                                               h->xi_int, h->cbuf.as<double>(), h->sflag.as<unsigned char>());
    SGPR_CUDA(cudaGetLastError());
    h->stats.kernel_launches += 1;
    return SGPR_OK;
}

}  // namespace

int descriptor_check_size(const DescParams& dp) {
    if ((size_t)plan_backward(dp).per_warp * 8 > 200 * 1024) {
        set_error("descriptor too large for shared memory (S=%d nmax=%d lmax=%d): the force kernel needs %zu KB per "
                  "warp, at most 200 KB fit", dp.S, dp.nb - 1, dp.lmax, (size_t)plan_backward(dp).per_warp * 8 / 1024);
        return SGPR_ERR_INVALID;
    }
    JacLayout lay;
    int nw;
    size_t smem;
    if (!plan_jacobian(dp, (dp.lmax <= 3 && dp.nb <= 4) ? 4 : 2, lay, nw, smem)) {   // MM of descriptor_jacobian_atoms
        set_error("descriptor too large for the Jacobian kernel (S=%d nmax=%d lmax=%d)", dp.S, dp.nb - 1, dp.lmax);
        return SGPR_ERR_INVALID;
    }
    return SGPR_OK;
}

int descriptor_jacobian_atoms(sgpr_context* h, const JacTarget& t, cudaStream_t st) {
    if (h->n_active == 0 || t.n_sel == 0) return SGPR_OK;
    EnvSrc src{};
    src.atoms = h->atoms.as<AtomRec>();
    src.pairs = h->nl_pairs.as<PairRec>();
    src.nl_rows = h->nl_rows.as<longlong2>();
    src.active = h->active_all ? nullptr : h->active_list.as<int>();
    JacArgs a{};
    a.sel = t.sel;
    a.sel_col = t.sel + t.n_sel;
    int max_sel = 0;
    for (int s = 0; s <= kMaxSpecies; ++s) a.sel_first[s] = t.sel_first[std::min(s, h->S)];
    for (int s = 0; s < h->S; ++s) max_sel = std::max(max_sel, t.sel_first[s + 1] - t.sel_first[s]);
    a.ncol = t.ncol;
    a.n_atoms = t.n_atoms;
    a.J = t.J;
    a.W = t.W;
    a.cells = t.cells;
    a.astr = t.astr;
    const int lmax = h->dp.lmax, nb = h->dp.nb;
#define JAC(LM, NBB, EX) return launch_jacobian<LM, NBB, EX>(h, src, a, max_sel, st)
    if (lmax == 3 && nb == 4) JAC(3, 4, true);   // the reference's default
    if (lmax <= 3 && nb <= 4) JAC(3, 4, false);
    if (lmax == 6 && nb == 9) JAC(6, 9, true);   // the high-resolution configuration
    if (lmax <= 3 && nb <= 8) JAC(3, 8, false);
    if (lmax <= 6 && nb <= 6) JAC(6, 6, false);
    if (lmax <= 6 && nb <= 9) JAC(6, 9, false);
    if (lmax <= 6 && nb <= 12) JAC(6, 12, false);
    if (lmax <= 8 && nb <= 12) JAC(8, 12, false);
#undef JAC
    set_error("unsupported descriptor size lmax=%d nmax=%d", lmax, nb - 1);
    return SGPR_ERR_INVALID;
}

int descriptor_forward_env(sgpr_context* h, int M, const long long* env_first_d, const double* env_r_d,
                           const unsigned char* env_sp_d, const int* row_of_d, double* phat_d, cudaStream_t st) {
    EnvSrc src{};
    src.env_first = env_first_d;
    src.env_r = env_r_d;
    src.env_sp = env_sp_d;
    Geom g{};
    return dispatch_forward<true>(h, g, M, src, row_of_d, phat_d, nullptr, nullptr, nullptr, st);
}

int descriptor_forward_atoms(sgpr_context* h, const Geom& g, cudaStream_t st, const BatchGeom* bg) {
    const int na = (int)h->n_active;
    const DescParams& dp = h->dp;
    SGPR_TRY(h->cbuf.ensure(sizeof(double) * ((size_t)na * dp.csize + 1)));
    SGPR_TRY(h->prow.ensure(sizeof(double) * ((size_t)na + 1)));
    SGPR_TRY(h->sflag.ensure((size_t)na + 1));
    if (na == 0) return SGPR_OK;
    EnvSrc src{};
    src.atoms = h->atoms.as<AtomRec>();
    src.pairs = h->nl_pairs.as<PairRec>();
    src.nl_rows = h->nl_rows.as<longlong2>();
    src.active = h->active_all ? nullptr : h->active_list.as<int>();
    if (bg)
        return dispatch_forward<false, true>(h, g, na, src, h->rowof.as<int>() + (h->last_N + 1), h->phat.as<double>(),
                                             h->cbuf.as<double>(), h->prow.as<double>(), h->sflag.as<unsigned char>(), st, bg);
    return dispatch_forward<false>(h, g, na, src, h->rowof.as<int>() + (h->last_N + 1), h->phat.as<double>(),
                                   h->cbuf.as<double>(), h->prow.as<double>(), h->sflag.as<unsigned char>(), st);
}

int backward_grid(sgpr_context* h) { return h->sm_count * 16; }

template <bool BATCH>
static int dispatch_backward(sgpr_context* h, const Geom& g, int na, const EnvSrc& src, const BackOut& out, cudaStream_t st,
                             const BatchGeom* bg) {
    const int grid = backward_grid(h);
    const int lmax = h->dp.lmax, nb = h->dp.nb;
#define BWD(LM, NBB) return launch_backward<LM, NBB, false, BATCH>(h, g, na, src, out, grid, st, bg)
    if (lmax == 3 && nb == 4) return launch_backward<3, 4, true, BATCH>(h, g, na, src, out, grid, st, bg);   // the reference's default
    if (lmax <= 3 && nb <= 4) BWD(3, 4);
    if (lmax == 6 && nb == 9) return launch_backward<6, 9, true, BATCH>(h, g, na, src, out, grid, st, bg);
    if (lmax <= 3 && nb <= 8) BWD(3, 8);
    if (lmax <= 6 && nb <= 6) BWD(6, 6);
    if (lmax <= 6 && nb <= 9) BWD(6, 9);
    if (lmax <= 6 && nb <= 12) BWD(6, 12);
    if (lmax <= 8 && nb <= 12) BWD(8, 12);
#undef BWD
    set_error("unsupported descriptor size lmax=%d nmax=%d", lmax, nb - 1);
    return SGPR_ERR_INVALID;
}

int descriptor_backward_atoms(sgpr_context* h, const Geom& g, const unsigned char* owned_d, cudaStream_t st,
                              const PeerForces* peers, const BatchGeom* bg) {
    const int na = (int)h->n_active;
    if (na == 0) return SGPR_OK;
    EnvSrc src{};
    src.atoms = h->atoms.as<AtomRec>();
    src.pairs = h->nl_pairs.as<PairRec>();
    src.nl_rows = h->nl_rows.as<longlong2>();
    src.active = h->active_all ? nullptr : h->active_list.as<int>();
    BackOut out{};
    if (peers) out.peers = *peers;
    out.fcell = (peers && peers->world > 0) ? peers->peer_f[h->p2p_rank] : h->fcell.as<double>();
    out.wpart = h->wpart.as<double>();
    out.owned = owned_d;
    out.sp_on = h->sp_on.as<unsigned char>();
    return bg ? dispatch_backward<true>(h, g, na, src, out, st, bg) : dispatch_backward<false>(h, g, na, src, out, st, nullptr);
}

int unpack_descriptors(sgpr_context* h, long long rows, const double* packed_d, const int* src_row_d, double* full_d,
                       cudaStream_t st) {
    if (rows == 0) return SGPR_OK;
    unpack_kernel<<<h->sm_count * 4, 256, 0, st>>>(h->dp, rows, packed_d, src_row_d, full_d);
    SGPR_CUDA(cudaGetLastError());
    h->stats.kernel_launches += 1;
    return SGPR_OK;
}

}  // namespace sgpr
