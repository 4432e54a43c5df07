// The two hot GEMMs of the prediction path on the 5th-generation tensor cores (tcgen05 + TMEM + TMA):
// float64-accurate through int8 digit slicing with exact int32 accumulation (i8gemm_kernel.cuh).
//
//   (1) kernel matrix   k[i,m] = q_hat_i . z_hat_m   (similarity/universal.py:109-122), epilogue:
//         e_i partials  sum_m mu_m k^xi               (calculator/active.py:548-550)
//         A2 = digits of k^(xi-1)                      (operand of the back projection)
//   (2) back projection g[i,:] = mumax * sum_m k^(xi-1)[i,m] * (xi mu_m z_hat_m / mumax)
//       = dE_i/dq_hat_i  (autograd through universal.py:121 in calculator/active.py:587-599)
//
// Operands: q_hat digits are written by the descriptor kernel, z_hat digits at sgpr_create,
// (xi mu z_hat^T / mumax) digits at sgpr_create / sgpr_set_weights.  All |values| <= 1 because the
// descriptors are normalised (|k| <= 1 by Cauchy-Schwarz); un-normalised models use the DMMA path.
#include <math.h>

#include "i8gemm_kernel.cuh"
#include "sgpr_internal.cuh"

namespace sgpr {

using namespace i8g;

namespace {

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn g_encode = nullptr;

int make_map(CUtensorMap* m, const void* base, int ns, long long rows, int Kpad, long long slice_stride_rows, int box_rows) {
    if (!g_encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
            set_error("cuTensorMapEncodeTiled is not available");
            return SGPR_ERR_CUDA;
        }
        g_encode = (EncodeFn)fn;
    }
    // K-chunk-major operand: element (slice t, row r, k) at  t * R * Kpad + (k / 64) * R * 64 + r * 64 + k % 64
    // with R = slice_stride_rows (the allocated rows); `rows` valid rows from `base` (out-of-range rows read as zero)
    cuuint64_t dims[4] = {64, (cuuint64_t)(rows > 0 ? rows : 1), (cuuint64_t)(Kpad / 64), (cuuint64_t)ns};
    cuuint64_t strides[3] = {64, (cuuint64_t)slice_stride_rows * 64, (cuuint64_t)slice_stride_rows * Kpad};
    cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, (cuuint32_t)ns};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(base), dims, strides, box, es,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): rows=%lld K=%d", (int)r, rows, Kpad);
        return SGPR_ERR_CUDA;
    }
    return SGPR_OK;
}

// Balanced base-256 digits of v = rint(x * 2^(8 NS - 2)):  v = sum_t d_t 256^t, d_t in [-128, 127].
// Adding the bias 128 * (1 + 256 + ... + 256^(NS-1)) makes every coefficient d_t + 128 lie in [0, 255],
// i.e. the bytes of (v + bias) ARE the digits + 128; xor 0x80 turns them into two's-complement int8.
template <int NS>
__device__ __forceinline__ unsigned long long digit_bytes(double x) {
    constexpr unsigned long long BIAS = 0x0080808080808080ull & ((1ull << (8 * NS)) - 1ull);
    // rint(x 2^(8 NS - 2)) without the 64-bit conversion unit: |x| <= 1, so adding 1.5 2^52 leaves the (round-to-nearest-
    // even) integer in the mantissa, offset by 2^51
    static_assert(8 * NS - 2 < 51, "the magic-number rounding needs |x 2^(8 NS - 2)| < 2^51");
    const long long v = __double_as_longlong(x * (double)(1ll << (8 * NS - 2)) + 6755399441055744.0) - 0x4338000000000000ll;
    return ((unsigned long long)(v + (long long)BIAS)) ^ BIAS;   // byte t = digit t (t = 0 least significant)
}
// byte b of four digit words -> one 32-bit word (columns j .. j+3 of one slice)
__device__ __forceinline__ unsigned gather_byte(const unsigned long long* u, int b) {
    unsigned w0, w1, w2, w3;
    if (b < 4) {
        w0 = (unsigned)u[0]; w1 = (unsigned)u[1]; w2 = (unsigned)u[2]; w3 = (unsigned)u[3];
    } else {
        w0 = (unsigned)(u[0] >> 32); w1 = (unsigned)(u[1] >> 32); w2 = (unsigned)(u[2] >> 32); w3 = (unsigned)(u[3] >> 32);
        b -= 4;
    }
    const unsigned sel = (unsigned)b | ((unsigned)(4 + b) << 4);
    const unsigned t01 = __byte_perm(w0, w1, sel), t23 = __byte_perm(w2, w3, sel);
    return __byte_perm(t01, t23, 0x5410);
}
template <int NS>
__device__ __forceinline__ void digits(double x, signed char* d) {   // most significant first
    const unsigned long long u = digit_bytes<NS>(x);
#pragma unroll
    for (int t = 0; t < NS; ++t) d[t] = (signed char)((u >> (8 * (NS - 1 - t))) & 0xff);
}

// float64 rows -> digit slices:  out[t][r][k] for r < rows, k < K ; zero for K <= k < Kpad
// chunk-major address of (row r, column k) inside one slice of an operand with R allocated rows
__host__ __device__ __forceinline__ long long cm_off(long long R, long long r, int k) {
    return (long long)(k >> 6) * (R * 64) + r * 64 + (k & 63);
}

template <int NS>
__global__ void slice_rows_kernel(const double* __restrict__ X, long long ldx, int rows, int K, int Kpad, double scale,
                                  const double* __restrict__ col_scale, signed char* __restrict__ out,
                                  long long slice_stride, const double* __restrict__ row_div = nullptr) {
    const long long R = slice_stride / Kpad;   // rows per slice
    const long long total = (long long)rows * Kpad;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(idx / Kpad), k = (int)(idx - (long long)r * Kpad);
        signed char d[NS];
        double x = 0.0;
        if (k < K) x = X[(long long)r * ldx + k] * scale * (col_scale ? col_scale[k] : 1.0);
        if (row_div) x /= row_div[r];   // power of two: exact
        digits<NS>(x, d);
#pragma unroll
        for (int t = 0; t < NS; ++t) out[(long long)t * slice_stride + cm_off(R, r, k)] = d[t];
    }
}

// power of two >= max |row| (1 for an all-zero row); one warp per row
__global__ void row_pow2_kernel(const double* __restrict__ X, long long ldx, int rows, int K, double* __restrict__ rs) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= rows) return;
    double m = 0.0;
    for (int k = lane; k < K; k += 32) m = fmax(m, fabs(X[(long long)r * ldx + k]));
    for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) {
        int e = 0;
        if (m > 0.0) frexp(m, &e);   // m = f 2^e, f in [0.5, 1)
        rs[r] = m > 0.0 ? ldexp(1.0, e) : 1.0;
    }
}

constexpr int kNS = 6;

// XI = 4 (the reference's default exponent): k^(xi-1) is two multiplies and nothing else is compiled in; XI = 0: any xi
template <int XI>
struct Epi1T {   // kernel matrix: energies + digits of k^(xi-1)
    double* erow_part;                   // [parts][erow_ld]
    signed char* g8;                     // slice 0, row 0
    signed char* k8;                     // digits of k^xi for the covloss GEMM (nullptr: not wanted)
    int erow_ld;
    int Mp;
    long long g8_slice;                  // bytes between slices
    long long cap_rows;                  // allocated rows of g8 / k8 (chunk-major layout)
    double xi;
    int xi_int;
    // mup (Problem::aux): mu of the species' inducing block
    __device__ void operator()(int p, int row0, int row, int col0, const double* v, int M, int N, const double* mup) const {
        if (row >= M) return;
        row += row0;
        double pw[16];
        // k^(xi-1): the usual exponents unrolled (independent multiplies), anything else by pow()
        if (XI == 4 || xi_int == 4) {
#pragma unroll
            for (int j = 0; j < 16; ++j) pw[j] = v[j] * v[j] * v[j];
        } else if (XI != 0) {
        } else if (xi_int == 2) {
#pragma unroll
            for (int j = 0; j < 16; ++j) pw[j] = v[j];
        } else if (xi_int == 3) {
#pragma unroll
            for (int j = 0; j < 16; ++j) pw[j] = v[j] * v[j];
        } else if (xi_int == 1) {
#pragma unroll
            for (int j = 0; j < 16; ++j) pw[j] = 1.0;
        } else {
#pragma unroll   // (a run-time index would put pw[] -- for every exponent -- into local memory)
            for (int j = 0; j < 16; ++j) {
                if (xi_int >= 1) {
                    double r = 1.0;
                    for (int t = 1; t < xi_int; ++t) r *= v[j];
                    pw[j] = r;
                } else {
                    pw[j] = pow(v[j], xi - 1.0);
                }
            }
        }
        double e = 0.0;
        unsigned long long u[16];
        if (col0 + 16 <= N) {   // whole chunk inside the matrix: no per-column masks
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                e += __ldg(mup + col0 + j) * pw[j] * v[j];
                u[j] = digit_bytes<kNS>(pw[j]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const bool in = col0 + j < N;
                const double pj = in ? pw[j] : 0.0;
                e += (in ? __ldg(mup + col0 + j) : 0.0) * pj * v[j];
                u[j] = digit_bytes<kNS>(pj);
            }
        }
        // one 16-byte store per slice (columns beyond N get zero digits: the K padding of GEMM 2)
        if (col0 < Mp) {
#pragma unroll
            for (int t = 0; t < kNS; ++t) {
                const int b = kNS - 1 - t;   // slice t (most significant first) = byte NS-1-t
                int4 w;
                w.x = (int)gather_byte(u + 0, b);
                w.y = (int)gather_byte(u + 4, b);
                w.z = (int)gather_byte(u + 8, b);
                w.w = (int)gather_byte(u + 12, b);
                *reinterpret_cast<int4*>(g8 + (long long)t * g8_slice + cm_off(cap_rows, row, col0)) = w;
            }
        }
        // energy partial of this 16-column chunk
        erow_part[(long long)(col0 >> 4) * erow_ld + row] = e;
        if (k8 != nullptr && col0 < Mp) {   // K = k^xi, the A operand of the covloss GEMM
#pragma unroll
            for (int j = 0; j < 16; ++j) u[j] = digit_bytes<kNS>(col0 + j < N ? pw[j] * v[j] : 0.0);
#pragma unroll
            for (int t = 0; t < kNS; ++t) {
                const int b = kNS - 1 - t;
                int4 w;
                w.x = (int)gather_byte(u + 0, b);
                w.y = (int)gather_byte(u + 4, b);
                w.z = (int)gather_byte(u + 8, b);
                w.w = (int)gather_byte(u + 12, b);
                *reinterpret_cast<int4*>(k8 + (long long)t * g8_slice + cm_off(cap_rows, row, col0)) = w;
            }
        }
    }
};

struct Epi3 {   // covloss: per-row partial sums of squares of b = K . choli^T  (calculator/active.py:781-783)
    double* part;                        // [parts][part_ld]
    int part_ld;
    // r (Problem::aux): power-of-two scales of the choli rows (= output columns)
    __device__ void operator()(int p, int row0, int row, int col0, const double* v, int M, int N, const double* r) const {
        if (row >= M) return;
        row += row0;
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const double t = col0 + j < N ? v[j] * r[col0 + j] : 0.0;
            s = fma(t, t, s);
        }
        part[(long long)(col0 >> 4) * part_ld + row] = s;
    }
};

struct Epi2 {   // back projection: g = mumax * C
    double* gvec;                        // [rows][ldp]
    int ldp;
    double mumax;
    __device__ void operator()(int p, int row0, int row, int col0, const double* v, int M, int N, const double*) const {
        if (row >= M) return;
        double* dst = gvec + (long long)(row0 + row) * ldp + col0;
        if (col0 + 16 <= N) {
#pragma unroll
            for (int j = 0; j < 16; j += 2) *reinterpret_cast<double2*>(dst + j) = make_double2(v[j] * mumax, v[j + 1] * mumax);
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if (col0 + j < N) dst[j] = v[j] * mumax;
        }
    }
};

template <int TR, int EPW = 2, class Epi>
int launch(sgpr_context* h, const Common* cm_d, const Problem* probs_d, const Epi& epi, cudaStream_t st) {
    constexpr int STAGES = 3;
    auto kern = i8gemm_kernel<kNS, TR, STAGES, Epi, 0, EPW>;
    const size_t smem = smem_bytes<kNS, STAGES>();
    static bool done = false;   // per instantiation
    if (!done) {
        SGPR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        done = true;
    }
    // persistent: one CTA per SM; the tile count lives on the device (CTAs beyond it exit at once)
    kern<<<h->sm_count, 64 + 128 * EPW, smem, st>>>(cm_d, probs_d, epi);
    SGPR_CUDA(cudaGetLastError());
    h->stats.kernel_launches += 1;
    return SGPR_OK;
}

// Work lists of the three grouped GEMMs from the species row ranges on the device (one warp).
typedef I8Setup SetupDesc;
__global__ void i8_setup_kernel(SetupDesc sd, const int* __restrict__ row_first, Common* __restrict__ out) {
    if (threadIdx.x >= 3) return;
    const int w = threadIdx.x;
    Common cm;
    cm.n_prob = sd.n_prob;
    int t = 0;
    for (int p = 0; p < 8; ++p) {
        cm.tile_start[p] = t;
        cm.row0[p] = 0;
        cm.M[p] = 0;
        if (p < sd.n_prob) {
            const int s = sd.species[p];
            const int r0 = row_first[s], r1 = row_first[s + 1];
            cm.row0[p] = r0;
            cm.M[p] = r1 - r0;
            t += ((r1 - r0 + BM - 1) / BM) * ((sd.ncol[w][p] + BN - 1) / BN);
        }
    }
    cm.tile_start[8] = t;
    // tile_start[n_prob] is the total the kernel reads
    for (int p = sd.n_prob; p < 9; ++p) cm.tile_start[p] = t;
    out[w] = cm;
}

}  // namespace

int i8_energy_parts(int Ms) { return ((Ms + BN - 1) / BN) * (BN / 16); }

// digit slices of the static operands: z_hat (GEMM 1) and xi mu z_hat^T / mumax (GEMM 2)
int i8_prepare_model(sgpr_context* h, bool weights_only) {
    const DescParams& dp = h->dp;
    const int M = h->M, S = h->S;
    h->i8_kp1 = (dp.D + 63) / 64 * 64;
    int maxMs = 0;
    for (int s = 0; s < S; ++s) maxMs = std::max(maxMs, h->m_first[s + 1] - h->m_first[s]);
    h->i8_mp = std::max(64, (maxMs + 63) / 64 * 64);
    h->i8_model_version++;
    if (M == 0) return SGPR_OK;
    if (!weights_only) {
        SGPR_TRY(h->z8.ensure((size_t)kNS * M * h->i8_kp1 + 64));
        slice_rows_kernel<kNS><<<h->sm_count * 4, 256>>>(h->zhat.as<double>(), dp.ldp, M, dp.D, h->i8_kp1, 1.0, nullptr,
                                                         h->z8.as<signed char>(), (long long)M * h->i8_kp1);
        SGPR_CUDA(cudaGetLastError());
    }
    // mumax: power of two >= max_m xi |mu_m|
    double mx = 0.0;
    for (double m : h->mu_host) mx = std::max(mx, std::fabs(h->xi * m));
    h->i8_mumax = mx > 0 ? std::ldexp(1.0, (int)std::ceil(std::log2(mx))) : 1.0;
    // per species: rows e of zhat_t [D, ld_zt], columns m scaled by xi mu_m / mumax
    SGPR_TRY(h->zt8.ensure((size_t)S * kNS * dp.D * h->i8_mp + 64));
    SGPR_CUDA(cudaMemset(h->zt8.p, 0, (size_t)S * kNS * dp.D * h->i8_mp));
    std::vector<double> cs(M + 1, 0.0);
    for (int p = 0; p < M; ++p) cs[p] = h->xi * h->mu_host[h->ind_perm[p]] / h->i8_mumax;
    SGPR_TRY(h->misc.ensure(sizeof(double) * (M + 1)));
    SGPR_CUDA(cudaMemcpy(h->misc.p, cs.data(), sizeof(double) * M, cudaMemcpyHostToDevice));
    for (int s = 0; s < S; ++s) {
        const int m0 = h->m_first[s], Ms = h->m_first[s + 1] - m0;
        if (Ms == 0) continue;
        slice_rows_kernel<kNS><<<h->sm_count * 4, 256>>>(h->zhat_t.as<double>() + h->zt_off[s], h->ld_zt, dp.D, Ms, h->i8_mp, 1.0,
                                                         h->misc.as<double>() + m0,
                                                         h->zt8.as<signed char>() + (size_t)s * kNS * dp.D * h->i8_mp,
                                                         (long long)dp.D * h->i8_mp);
        SGPR_CUDA(cudaGetLastError());
    }
    SGPR_CUDA(cudaDeviceSynchronize());
    return SGPR_OK;
}

// digit slices of choli for the covloss GEMM: per central species s the rows k of choli[:, columns of s]
// (h->choli_t), each divided by its own power-of-two bound so that small rows keep their relative accuracy
int i8_prepare_covloss(sgpr_context* h) {
    const int M = h->M, S = h->S;
    if (M == 0 || !h->has_choli) return SGPR_OK;
    SGPR_TRY(h->crs.ensure(sizeof(double) * (size_t)S * M));
    SGPR_TRY(h->c8.ensure((size_t)S * kNS * M * h->i8_mp + 64));
    SGPR_CUDA(cudaMemset(h->c8.p, 0, (size_t)S * kNS * M * h->i8_mp));
    for (int s = 0; s < S; ++s) {
        const int Ms = h->m_first[s + 1] - h->m_first[s];
        if (Ms == 0) continue;
        const double* X = h->choli_t.as<double>() + (size_t)s * M * h->ld_zt;
        double* rs = h->crs.as<double>() + (size_t)s * M;
        row_pow2_kernel<<<(M + 7) / 8, 256>>>(X, h->ld_zt, M, Ms, rs);
        slice_rows_kernel<kNS><<<h->sm_count * 4, 256>>>(X, h->ld_zt, M, Ms, h->i8_mp, 1.0, nullptr,
                                                         h->c8.as<signed char>() + (size_t)s * kNS * M * h->i8_mp,
                                                         (long long)M * h->i8_mp, rs);
        SGPR_CUDA(cudaGetLastError());
    }
    SGPR_CUDA(cudaDeviceSynchronize());
    // K extent per (species, 64-column tile): choli = L^-1 is lower triangular (regression/gppotential.py:588), so
    // for output columns k only inducing LCEs m <= k contribute; chunks beyond the last non-zero are never loaded
    {
        const int ntn = (M + BN - 1) / BN;
        std::vector<double> host((size_t)S * M * h->ld_zt);
        SGPR_CUDA(cudaMemcpy(host.data(), h->choli_t.p, sizeof(double) * host.size(), cudaMemcpyDeviceToHost));
        std::vector<int> nk((size_t)S * ntn, 0);
        for (int s = 0; s < S; ++s) {
            const int Ms = h->m_first[s + 1] - h->m_first[s];
            for (int tn = 0; tn < ntn; ++tn) {
                int ext = 0;
                for (int k = tn * BN; k < std::min(M, (tn + 1) * BN); ++k) {
                    const double* row = host.data() + ((size_t)s * M + k) * h->ld_zt;
                    for (int p = Ms - 1; p >= ext; --p)
                        if (row[p] != 0.0) {
                            ext = p + 1;
                            break;
                        }
                }
                nk[(size_t)s * ntn + tn] = (ext + BKB - 1) / BKB;   // 0: the tile is identically zero
            }
        }
        SGPR_TRY(h->cov_nk.ensure(sizeof(int) * nk.size()));
        SGPR_CUDA(cudaMemcpy(h->cov_nk.p, nk.data(), sizeof(int) * nk.size(), cudaMemcpyHostToDevice));
    }
    return SGPR_OK;
}

// buffers written by the descriptor kernel (q_hat digits) and by GEMM 1 (k^(xi-1) and, for covloss, k^xi digits)
int i8_ensure_step_buffers(sgpr_context* h, size_t n_rows, bool with_k8) {
    const size_t cap = n_rows + 1;
    if (with_k8) SGPR_TRY(h->k8.ensure((size_t)kNS * std::max(h->i8_cap_rows, cap + cap / 4) * h->i8_mp + 64));
    if (cap > h->i8_cap_rows) {
        const size_t c = cap + cap / 4;
        SGPR_TRY(h->p8.ensure((size_t)kNS * c * h->i8_kp1 + 64));
        SGPR_TRY(h->g8.ensure((size_t)kNS * c * h->i8_mp + 64));
        // pad columns of p8 (D <= k < Kp1) are never written by the descriptor kernel: keep them zero
        SGPR_CUDA(cudaMemset(h->p8.p, 0, (size_t)kNS * c * h->i8_kp1));
        h->i8_cap_rows = c;
    }
    return SGPR_OK;
}

// Problem descriptors (tensor maps over the WHOLE operand buffers + static shapes) of GEMM `which`; they depend only on
// the model and on the buffer addresses, not on the step: rebuilt and uploaded when those change.
static int build_problems(sgpr_context* h, int which, std::vector<Problem>& probs, SetupDesc& sd) {
    const DescParams& dp = h->dp;
    probs.clear();
    sd.n_prob = 0;
    const long long cap = (long long)h->i8_cap_rows;
    for (int s = 0; s < h->S; ++s) {
        const int m0 = h->m_first[s], m1 = h->m_first[s + 1];
        if (m1 == m0 || !dp.central_enabled[s]) continue;
        Problem P;
        P.nk_tn = nullptr;
        P.aux = nullptr;
        P.M = 0;
        if (which == 1) {
            P.aux = h->mu.as<double>() + m0;
            P.N = m1 - m0;
            P.Kpad = h->i8_kp1;
            SGPR_TRY(make_map(&P.mapA, h->p8.as<signed char>(), kNS, cap, P.Kpad, cap, BM));
            SGPR_TRY(make_map(&P.mapB, h->z8.as<signed char>() + (size_t)m0 * 64, kNS, P.N, P.Kpad, (long long)h->M, BN));
        } else if (which == 2) {
            P.N = dp.D;
            P.Kpad = ((m1 - m0) + 63) / 64 * 64;
            SGPR_TRY(make_map(&P.mapA, h->g8.as<signed char>(), kNS, cap, h->i8_mp, cap, BM));
            SGPR_TRY(make_map(&P.mapB, h->zt8.as<signed char>() + (size_t)s * kNS * dp.D * h->i8_mp, kNS, dp.D, h->i8_mp, (long long)dp.D, BN));
        } else {
            P.aux = h->crs.as<double>() + (size_t)s * h->M;
            P.N = h->M;
            P.Kpad = ((m1 - m0) + 63) / 64 * 64;
            SGPR_TRY(make_map(&P.mapA, h->k8.as<signed char>(), kNS, cap, h->i8_mp, cap, BM));
            SGPR_TRY(make_map(&P.mapB, h->c8.as<signed char>() + (size_t)s * kNS * h->M * h->i8_mp, kNS, h->M, h->i8_mp, (long long)h->M, BN));
            const int ntn = (h->M + BN - 1) / BN;
            if (h->cov_nk.p) P.nk_tn = h->cov_nk.as<int>() + (size_t)s * ntn;
        }
        sd.species[sd.n_prob] = s;
        sd.ncol[0][sd.n_prob] = m1 - m0;
        sd.ncol[1][sd.n_prob] = dp.D;
        sd.ncol[2][sd.n_prob] = h->M;
        sd.n_prob++;
        probs.push_back(P);
    }
    return SGPR_OK;
}

// algorithmic work of the step's GEMMs (needs the species row ranges on the host: sizing steps only)
static void count_work(sgpr_context* h, int which) {
    const DescParams& dp = h->dp;
    if (!h->row_first_host_valid) return;
    for (int s = 0; s < h->S; ++s) {
        const int r0 = h->row_first[s], r1 = h->row_first[s + 1];
        const int m0 = h->m_first[s], m1 = h->m_first[s + 1];
        if (r1 == r0 || m1 == m0 || !dp.central_enabled[s]) continue;
        const double M = r1 - r0;
        if (which == 3) {
            // algorithmic flops of the dense product; the zero part of a triangular choli is skipped, not counted less
            h->stats.covloss_flops += 2.0 * M * (double)h->M * (m1 - m0);
        } else {
            const int tr = which == 2 ? h->i8_tr2 : h->i8_tr;
            const int npairs = tr == 8 ? 26 : 21;
            const double N = which == 1 ? (m1 - m0) : dp.D;
            const double Kpad = which == 1 ? h->i8_kp1 : ((m1 - m0) + 63) / 64 * 64;
            h->stats.gemm_flops += 2.0 * M * N * (which == 1 ? dp.D : (m1 - m0));
            h->stats.i8_ops += 2.0 * M * N * Kpad * npairs;
        }
    }
}

// Problems of GEMM `which` on the device (slot which-1), re-uploaded only when the model or a buffer moved.
static int device_problems(sgpr_context* h, int which, cudaStream_t st, const Problem** out, SetupDesc* sd_out) {
    SGPR_TRY(h->i8_probs.ensure(sizeof(Problem) * 3 * kMaxSpecies + sizeof(Common) * 4));
    if (!h->i8_probs_pinned) SGPR_CUDA(cudaMallocHost(&h->i8_probs_pinned, sizeof(Problem) * 3 * kMaxSpecies));
    const int slot = which - 1;
    // signature of everything the descriptors encode
    unsigned long long sig = 1469598103934665603ull;
    auto mix = [&](unsigned long long v) { sig = (sig ^ v) * 1099511628211ull; };
    mix((unsigned long long)(uintptr_t)h->p8.p); mix((unsigned long long)(uintptr_t)h->g8.p); mix((unsigned long long)(uintptr_t)h->k8.p);
    mix((unsigned long long)(uintptr_t)h->z8.p); mix((unsigned long long)(uintptr_t)h->zt8.p); mix((unsigned long long)(uintptr_t)h->c8.p);
    mix((unsigned long long)(uintptr_t)h->cov_nk.p); mix((unsigned long long)(uintptr_t)h->i8_probs.p);
    mix((unsigned long long)(uintptr_t)h->mu.p); mix((unsigned long long)(uintptr_t)h->crs.p);
    mix(h->i8_cap_rows); mix(h->M); mix(h->i8_kp1); mix(h->i8_mp); mix(h->i8_model_version);
    for (int s = 0; s <= h->S; ++s) mix(h->m_first[s]);
    Problem* dev = h->i8_probs.as<Problem>() + slot * kMaxSpecies;
    if (h->i8_prob_sig[slot] != sig) {
        std::vector<Problem> probs;
        SetupDesc sd{};
        SGPR_TRY(build_problems(h, which, probs, sd));
        Problem* pin = (Problem*)h->i8_probs_pinned + slot * kMaxSpecies;
        // the staging slot may still be read by an earlier asynchronous upload
        SGPR_CUDA(cudaStreamSynchronize(st));
        for (size_t i = 0; i < probs.size(); ++i) pin[i] = probs[i];
        if (!probs.empty()) SGPR_CUDA(cudaMemcpyAsync(dev, pin, sizeof(Problem) * probs.size(), cudaMemcpyHostToDevice, st));
        h->i8_prob_sig[slot] = sig;
        h->i8_setup[slot] = sd;
    }
    *out = dev;
    *sd_out = h->i8_setup[slot];
    return SGPR_OK;
}

static Common* common_d(sgpr_context* h, int which) {
    return reinterpret_cast<Common*>(h->i8_probs.as<Problem>() + 3 * kMaxSpecies) + (which - 1);
}

// one-warp set-up kernel: the three work lists of this step from the device-side species row ranges
int i8_setup_step(sgpr_context* h, cudaStream_t st) {
    const Problem* dummy = nullptr;
    SetupDesc sd{};
    SGPR_TRY(device_problems(h, 1, st, &dummy, &sd));
    if (sd.n_prob == 0) {
        h->i8_nprob = 0;
        return SGPR_OK;
    }
    h->i8_nprob = sd.n_prob;
    i8_setup_kernel<<<1, 32, 0, st>>>(sd, h->row_first_d.as<int>(), common_d(h, 1));
    SGPR_CUDA(cudaGetLastError());
    h->stats.kernel_launches += 1;
    return SGPR_OK;
}

template <class Epi1>
static int kernel_matrix_impl(sgpr_context* h, cudaStream_t st, bool store_k8, const Problem* probs_d, const SetupDesc& sd) {
    Epi1 e{};
    e.erow_part = h->erow_part.as<double>();
    e.g8 = h->g8.as<signed char>();
    e.k8 = store_k8 ? h->k8.as<signed char>() : nullptr;
    e.erow_ld = (int)h->n_active + 1;
    e.Mp = h->i8_mp;
    e.g8_slice = (long long)h->i8_cap_rows * h->i8_mp;
    e.cap_rows = (long long)h->i8_cap_rows;
    e.xi = h->xi;
    e.xi_int = h->xi_int;
    // descriptors of one K chunk (a single species with the default lmax/nmax): the main loop is one stage per tile and
    // the fused epilogue is the kernel -- twice the epilogue warps
    if (h->i8_tr == 7 && h->i8_kp1 <= 64) return launch<7, 4>(h, common_d(h, 1), probs_d, e, st);
    return h->i8_tr == 8 ? launch<8>(h, common_d(h, 1), probs_d, e, st) : launch<7>(h, common_d(h, 1), probs_d, e, st);
}

int i8_kernel_matrix(sgpr_context* h, cudaStream_t st, bool store_k8) {
    const Problem* probs_d = nullptr;
    SetupDesc sd{};
    SGPR_TRY(device_problems(h, 1, st, &probs_d, &sd));
    if (sd.n_prob == 0) return SGPR_OK;
    count_work(h, 1);
    if (h->xi_int == 4) return kernel_matrix_impl<Epi1T<4>>(h, st, store_k8, probs_d, sd);
    return kernel_matrix_impl<Epi1T<0>>(h, st, store_k8, probs_d, sd);
}

int i8_back_projection(sgpr_context* h, cudaStream_t st) {
    const Problem* probs_d = nullptr;
    SetupDesc sd{};
    SGPR_TRY(device_problems(h, 2, st, &probs_d, &sd));
    if (sd.n_prob == 0) return SGPR_OK;
    count_work(h, 2);
    Epi2 e{};
    e.gvec = h->gvec.as<double>();
    e.ldp = h->dp.ldp;
    e.mumax = h->i8_mumax;
    return h->i8_tr2 == 8 ? launch<8>(h, common_d(h, 2), probs_d, e, st) : launch<7>(h, common_d(h, 2), probs_d, e, st);
}

// Covloss GEMM on tcgen05: b = K . choli^T per central species, reduced on the fly to per-row partial sums of
// squares (h->cpart [i8_covloss_parts, n_rows]).  Always 26 slice products (t + u <= 8): choli is not normalised.
int i8_covloss_parts(sgpr_context* h) { return ((h->M + BN - 1) / BN) * (BN / 16); }

int i8_covloss(sgpr_context* h, int64_t n_rows, cudaStream_t st) {
    const Problem* probs_d = nullptr;
    SetupDesc sd{};
    SGPR_TRY(device_problems(h, 3, st, &probs_d, &sd));
    if (sd.n_prob == 0) return SGPR_OK;
    count_work(h, 3);
    Epi3 e{};
    e.part = h->cpart.as<double>();
    e.part_ld = (int)n_rows;
    return launch<8>(h, common_d(h, 3), probs_d, e, st);
}

}  // namespace sgpr
