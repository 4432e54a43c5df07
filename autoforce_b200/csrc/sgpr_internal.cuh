// Internal declarations shared by the translation units of libsgpr_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <functional>
#include <string>
#include <vector>

#include "../../include/sgpr_b200.h"
#include "sgpr_math.cuh"

#define SGPR_MAX_RANKS 16

namespace sgpr {

// ----------------------------------------------------------------------------------
// errors
// ----------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define SGPR_CUDA(call)                                                                    \
    do {                                                                                   \
        cudaError_t _e = (call);                                                           \
        if (_e != cudaSuccess) {                                                           \
            sgpr::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return SGPR_ERR_CUDA;                                                          \
        }                                                                                  \
    } while (0)
#define SGPR_TRY(call)                \
    do {                              \
        int _s = (call);              \
        if (_s != SGPR_OK) return _s; \
    } while (0)

// ----------------------------------------------------------------------------------
// device-side views
// ----------------------------------------------------------------------------------

// Atom record in cell order: position as given by the caller (NOT wrapped) + meta word.
//   meta bits  0..31 original index | 32..39 species index | 40..47 w0+128 | 48..55 w1+128
//              | 56..63 w2+128      (w = floor(frac) on periodic axes: wrap shift)
struct __align__(32) AtomRec {
    double x, y, z;
    unsigned long long meta;
};
__host__ __device__ inline int meta_orig(unsigned long long m) { return (int)(m & 0xffffffffull); }
__host__ __device__ inline int meta_species(unsigned long long m) { return (int)((m >> 32) & 0xff); }
__host__ __device__ inline int meta_w(unsigned long long m, int c) { return (int)((m >> (40 + 8 * c)) & 0xff) - 128; }

// Neighbour pair record (8 bytes): cell-order index of j, bin-level image shift
// (relative to WRAPPED positions) and species of j.
struct __align__(8) PairRec {
    int j;
    signed char sb[3];
    unsigned char sp;
};

struct Geom {
    double cell[9];   // rows = lattice vectors (completed on non-periodic axes)
    double inv[9];    // frac_c = sum_k pos_k * inv[k*3+c]
    double flo[3];    // non-periodic axes: lower bound of frac coordinate
    double fscale[3]; // bin = floor((frac - flo) * fscale)
    int pbc[3];
    int nb[3];        // bins per axis
    int reach[3];     // stencil reach per axis
    int ncell;
    double rc;
};

// Everything the descriptor kernels need to know about the model (passed by value).
struct DescParams {
    int lmax, nb;           // nb = nmax+1
    int L2;                 // (lmax+1)^2
    int L2p;                // row stride of c[a][lm] (L2 made odd: conflict-free smem columns)
    int S;                  // species
    int A;                  // S*nb
    int ncomp;              // nb*L2  (components per species)
    int csize;              // A*L2p  (padded expansion-coefficient block per atom)
    int D;                  // packed descriptor length = A(A+1)/2*(lmax+1)
    int ldp;                // leading dimension of packed descriptor rows (doubles)
    int normalize;
    double rc;
    double rc_inv;                  // 1 / rc
    double radii[kMaxSpecies];
    double rinv[kMaxSpecies];       // 1 / radii (exact for the reference's radii 1.0 and 0.5)
    int central_enabled[kMaxSpecies];
    int nbr_enabled[kMaxSpecies];   // 0: neighbours of this species are left out of the expansion
};

// static part of the grouped tcgen05 GEMM work lists (i8gemm.cu): which central species form a problem and how many
// output columns each has in GEMM 1 (kernel matrix), 2 (back projection), 3 (covloss)
struct I8Setup {
    int n_prob;
    int species[kMaxSpecies];
    int ncol[3][kMaxSpecies];
};

// Batched prediction (sgpr_predict_batch): per-structure geometry and indices, device pointers.  Structure b holds the
// atoms first[b] .. first[b+1]-1 of the caller's order and, because the cell-sort keys are structure-major, the same
// index range of the cell order; its bins are bin_base[b] .. bin_base[b+1]-1 of the batch's bin table.
struct BatchGeom {
    int B;
    int ncell;                 // bins of the whole batch
    const Geom* geoms;         // [B]   what build_geometry gives each structure alone
    const long long* first;    // [B+1] atom offsets
    const int* bin_base;       // [B+1]
    const double* cells;       // [B,9] completed cells (image shifts of the descriptor kernels)
    int* astr;                 // [N]   structure of cell-order atom c
    unsigned long long* err;   // [2]   min (b << 32 | Z) over unknown species, min b over atoms too far outside their cell
};

// Number of DevBuf reallocations so far: CUDA graphs of warm steps bake the workspaces' addresses into their nodes and
// must not outlive them (api.cu: predict_impl).
unsigned long long buf_generation();

// max that propagates NaN, like torch.max / np.max in prediction mode (the device drivers' reductions)
__device__ __forceinline__ double nan_max(double a, double b) { return (b > a || b != b) ? b : a; }

// host-side mirror of a grow-only device buffer
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need);  // returns sgpr_status
    void release();
    template <class T> T* as() const { return (T*)p; }
};

}  // namespace sgpr

// ----------------------------------------------------------------------------------
// the handle
// ----------------------------------------------------------------------------------
struct sgpr_context {
    int device = 0;
    int sm_count = 148;
    // ---- model (host copies)
    sgpr::DescParams dp;
    double xi = 4.0;
    int xi_int = 4;                          // xi when it is a small positive integer, else -1
    int S = 0;
    int species_Z[SGPR_MAX_SPECIES];
    int z_to_species[128];                   // atomic number -> species index or -1
    int M = 0;
    int m_first[SGPR_MAX_SPECIES + 1];       // inducing LCEs grouped by central species (sorted order)
    int ld_zt = 0;                           // leading dim of the transposed Z_hat blocks
    int ldg = 0;                             // leading dim of G
    size_t zt_off[SGPR_MAX_SPECIES];         // offset (doubles) of species s inside zhat_t
    std::vector<int> ind_perm;               // sorted position -> caller's inducing index
    std::vector<int> ind_sp;                 // species of sorted inducing p
    std::vector<unsigned char> ind_lone;     // sorted inducing p has no neighbours
    std::vector<double> mean_w, vscale, mu_host;
    double lone_w = 1.0;        // weight of the lone-lone kernel term (number of similarity kernels)
    bool has_choli = false;
    std::vector<int32_t> ind_Z_host, ind_b_host;   // inducing environments as given (for sgpr_append_inducing)
    std::vector<int64_t> ind_first_host;
    std::vector<double> ind_r_host;
    // ---- model (device)
    sgpr::DevBuf zhat;        // [M, ldp]  packed normalised descriptors, rows grouped by species
    sgpr::DevBuf zhat_t;      // [S][D, ld_zt]  per-species transposes
    sgpr::DevBuf mu;          // [M] sorted order
    sgpr::DevBuf lone_mu;     // [S] sum of mu over neighbour-less inducing LCEs of species s
    sgpr::DevBuf mean_w_d;    // [S]
    sgpr::DevBuf choli_t;     // [S][M, ld_zt]: choli[:, columns of species s] (sorted order), zero padded
    sgpr::DevBuf vscale_d;    // [S] model._vscale (inf where unseen)
    sgpr::DevBuf clone_d;     // [S] c of a neighbour-less atom of species s
    sgpr::DevBuf kcmat, cpart;  // covloss: K^xi [rows, ldg], per-row partial sums of squares
    sgpr::DevBuf erow_part, erow, prow;  // per-row energy partials / local energies / descriptor norms
    sgpr::DevBuf ttab;          // [D] kappa*nnl*(1 + [a==b]) per packed entry
    // ---- tcgen05 int8-sliced GEMM path (i8gemm.cu)
    bool nl_lean = true;        // SGPR_NL_LEAN=0: force the many-kernel cell sort / row scan that very large systems use -- test hook
    int nl_mode = 0;            // SGPR_NL: 0 auto, 1 "warp" (one warp per environment), 2 "bins" (one block per bin) -- test hook
    sgpr::DevBuf nl_run;        // running per-species fill offsets across candidate tiles (block-per-bin fill)
    bool use_i8 = false;        // GEMMs on tcgen05 (int8 digit slices) instead of FP64 DMMA
    bool use_i8_now = false;    // ... for the current call (compat / K-matrix calls use the DMMA path)
    int i8_tr = 7;              // kernel matrix: truncation t + u <= i8_tr (7: 21 slice products, 8: 26)
    int i8_tr2 = 7;             // back projection: 7 / 8, or 6 (SGPR_I8_TR2=6: 15 products of 5 slices, ~4e-11 mumax on dE/dq_hat)
    int i8_ns = 6;              // digit slices read by the GEMMs with t + u <= 7 (SGPR_I8_NS=5: the 5 most significant of the
                                // 6 stored: 19 products, 38-bit operands)
    int i8_kp1 = 0, i8_mp = 0;  // K paddings (multiples of 64) of GEMM 1 (D) and GEMM 2 (max M_s)
    size_t i8_cap_rows = 0;     // row capacity of p8 / g8 (slice stride)
    double i8_mumax = 1.0;      // power of two >= max xi |mu|
    sgpr::DevBuf z8, zt8;       // static digit slices: z_hat [6][M][kp1], (xi mu z_hat^T / mumax) [S][6][D][mp]
    sgpr::DevBuf p8, g8;        // per-step digit slices: q_hat [6][cap][kp1], k^(xi-1) [6][cap][mp]
    sgpr::DevBuf cov_nk;        // [S][ceil(M/64)] non-zero K chunks of choli per column tile (triangular skip)
    sgpr::DevBuf k8, c8, crs;   // covloss: k^xi digits [6][cap][mp], choli digits [S][6][M][mp], choli row scales [S][M]
    sgpr::DevBuf i8_probs;      // device copies of the tensor-map problem descriptors + the three per-step work lists
    void* i8_probs_pinned = nullptr;
    unsigned long long i8_prob_sig[3] = {0, 0, 0};   // what the uploaded descriptors were built from (addresses, shapes)
    sgpr::I8Setup i8_setup[3];
    int i8_nprob = 0;
    int i8_epw = 0;              // SGPR_I8_EPW=2: never use the 4-epilogue-warps-per-quarter kernel (A/B switch)
    bool i8_cta2 = false;        // SGPR_I8_CTA2=1: CTA-pair (cta_group::2) variant of the two hot GEMMs
    sgpr::DevBuf i8_probs2;      // its problem descriptors
    void* i8_probs2_pinned = nullptr;
    unsigned long long i8_prob2_sig[2] = {0, 0};
    unsigned long long i8_model_version = 0;
    // ---- species row ranges / pair count stay on the device (sync-free steps, DESIGN.md section 4.2)
    sgpr::DevBuf row_first_d;   // [S+1] first descriptor row of each central species (device copy of row_first)
    bool row_first_host_valid = false;   // h->row_first[] describes the current step (sizing steps only)
    sgpr::DevBuf status_d;      // [8] long long: 0 pairs of the step, 1 sticky count of invalid steps, 2-5 error flags
    long long* status_pinned = nullptr;  // host mirror, copied at the end of a step
    long long pairs_cap = 0;    // capacity of nl_pairs (records)
    bool warm_ok = false;       // sizes of a previous step are valid: the next one may run without host synchronisation
    int64_t warm_N = -1;
    int warm_rank = -1, warm_world = -1;
    bool warm_halo = false;
    bool async_mode = false;    // sgpr_set_async: device-pointer entry points skip the sizing synchronisation when warm
    bool step_was_warm = false;
    long long bad_steps_seen = 0;   // value of the sticky invalid-step counter already reported
    bool warm_beta = false;
    // ---- CUDA graphs of warm steps (api.cu: predict_impl), keyed by everything baked into the nodes
    struct GraphKey {
        int64_t N;
        int rank, world;
        void* stream;
        const void* ptr[7];                 // pos, Z, E, F, W, beta, owned
        uint64_t peer[SGPR_MAX_RANKS];      // peer force buffers (p2p exchange)
        double cell[9];
        long long px_on;                    // fused exchange step
        const void* px_ptr[3];
        uint64_t px_mail[SGPR_MAX_RANKS];
    };
    struct GraphEntry {
        GraphKey key;
        cudaGraphExec_t exec;
        unsigned long long stamp;
        long long launches;
    };
    std::vector<GraphEntry> graphs;
    unsigned long long graph_clock = 0;
    unsigned long long graph_gen = 0;   // sgpr::buf_generation() the graphs were captured under
    bool use_graph = true;          // SGPR_GRAPH=0 switches the replay off
    sgpr::DevBuf ptab, nnlk;  // packed-entry tables [D]
    sgpr::DevBuf ztab;        // [128] atomic number -> species
    sgpr::DevBuf ind_perm_d;  // [M]
    sgpr::DevBuf ind_sp_d, ind_lone_d;  // [M] caller's order (lone-lone kernel term)
    sgpr::DevBuf sp_on;       // [S] species has usable inducing points and is enabled as a centre
    sgpr::DevBuf errflag;     // [4] ints
    // ---- per-call workspaces (grow-only)
    sgpr::DevBuf cnt, cstart, rstart, keyrank, atoms, order, rowof, active_list, rowmap;
    sgpr::DevBuf nl_cnt, nl_first, nl_pairs, nl_masks, scan_tmp;
    sgpr::DevBuf owned, shard_tmp, row_owned;    // atom sharding: owned/mark masks, scans, per-row ownership
    sgpr::DevBuf phat, cbuf, pnorm, sflag, gmat, gvec, epart, wpart, fcell, misc;
    sgpr::DevBuf stage_pos, stage_z, stage_out;  // device staging for the host API
    sgpr::DevBuf p2p_local;                      // fused exchange step: [16] partial E/W + step counter
    sgpr::DevBuf b_geom, b_first, b_bins, b_cell, b_err;   // batched prediction: BatchGeom arrays
    sgpr::DevBuf astr, wenv;                     // batched prediction: structure per cell-order atom, [N,9] per-environment virials
    sgpr::DevBuf jsel, kscr;                     // training-time kernels: inducing selection, K scratch [N, M]
    bool p2p_counter_init = false;
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
    cudaStream_t own_stream = nullptr;
    // ---- state of the current / last call
    int64_t last_N = 0;
    int64_t n_active = 0;
    int64_t n_owned = 0;
    bool active_all = true;
    int p2p_rank = 0;                        // this rank in a peer-memory force exchange
    bool fwd_valid = false;                  // state of the last sgpr_kernel_forward is intact (for the VJP)
    int row_first[SGPR_MAX_SPECIES + 1];     // first descriptor row of each central species
    sgpr::Geom last_geom;
    sgpr_stats stats;
    bool timing = false;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // ---- MD driver (md.cu): the step in flight is predicted from scratch copies and committed only when it was valid
    sgpr::DevBuf md_pos, md_mom, md_F, md_beta, md_ew, md_part;
    // ---- relaxation driver (relax.cu), same rule: scratch positions (first the step dr), velocities, forces, beta
    sgpr::DevBuf rx_pos, rx_vel, rx_F, rx_beta, rx_ew, rx_part;
    // ---- CUDA graphs of warm driver steps (md.cu: driver_graph_step), MD and relaxation in one LRU cache
    struct DriverGraphKey {                 // everything a captured driver step bakes into its nodes
        int32_t driver;                     // kDriverMd / kDriverRelax: keeps the two drivers' graphs apart
        int32_t flag[3];
        int64_t N;
        void* stream;
        const void* ptr[10];
        double cell[9];
        double prm[10];
        uint64_t seed;
    };
    struct DriverGraphEntry {
        DriverGraphKey key;
        cudaGraphExec_t exec;
        unsigned long long stamp;
    };
    std::vector<DriverGraphEntry> driver_graphs;
    unsigned long long driver_graph_gen = 0;
};

namespace sgpr {

// ---- nl.cu ------------------------------------------------------------------------
int build_geometry(sgpr_context* h, int64_t N, const double* pos_d, const double* cell_h, const int32_t* pbc_h,
                   cudaStream_t st, Geom* g);
// every structure's Geom as build_geometry gives it alone (one segmented bounds kernel, one synchronisation when a
// structure is not periodic on all axes)
int build_geometry_batch(sgpr_context* h, int B, const int64_t* first_h, const double* pos_d, const double* cell_h,
                         const int32_t* pbc_h, cudaStream_t st, std::vector<Geom>* gs);
// structure-major cell sort + neighbour list of all atoms of a batch (sizing: synchronises the stream)
int batch_cell_sort(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const BatchGeom& bg, cudaStream_t st);
int batch_neighbor_build(sgpr_context* h, int64_t N, const BatchGeom& bg, cudaStream_t st, int64_t* n_pairs);
int cell_sort(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const Geom& g, cudaStream_t st);
// warm = true: no device-to-host copy, no synchronisation -- pair count, error flags and species row ranges stay on
// the device (status_d, row_first_d); needs h->pairs_cap from an earlier sizing step; *n_pairs is then not set
int neighbor_build(sgpr_context* h, int64_t N, const Geom& g, cudaStream_t st, int64_t* n_pairs, bool warm = false);
int neighbor_build_sharded(sgpr_context* h, int64_t N, const Geom& g, int rank, int world, cudaStream_t st,
                           int64_t* n_pairs, bool with_halo = true, bool warm = false);
int scan_exclusive_ll(sgpr_context* h, const long long* in, long long* out, int n, cudaStream_t st);

// ---- descriptor.cu ----------------------------------------------------------------
int upload_harm_coef();
// refuses (SGPR_ERR_INVALID, message set) a descriptor size whose shared-memory plans of the force or Jacobian kernel
// cannot fit one warp
int descriptor_check_size(const DescParams& dp);
int descriptor_forward_env(sgpr_context* h, int M, const long long* env_first_d, const double* env_r_d,
                           const unsigned char* env_sp_d, const int* row_of_d, double* phat_d, cudaStream_t st);
int descriptor_forward_atoms(sgpr_context* h, const Geom& g, cudaStream_t st, const BatchGeom* bg = nullptr);
// peer-memory force exchange: neighbour forces go to the owner rank's buffer (peer_f[r] valid on this device)
struct PeerForces {
    double* peer_f[SGPR_MAX_RANKS];
    int bounds[SGPR_MAX_RANKS + 1];   // first cell-order index owned by each rank
    int world;                        // 0 = disabled
    // fused exchange step: two accumulation buffers per rank alternate between steps; WHICH one is decided on the
    // device (low bit of the step counter), so that the launch arguments -- and the CUDA graph -- never change
    const long long* parity_src;      // nullptr: peer_f as given
    long long parity_stride;          // doubles between the two buffers
};
// bg: batched step -- image shifts from the centre's structure, per-environment virials into h->wenv [N,9]
int descriptor_backward_atoms(sgpr_context* h, const Geom& g, const unsigned char* owned_d, cudaStream_t st,
                              const PeerForces* peers = nullptr, const BatchGeom* bg = nullptr);
// fused exchange step (api.cu: sgpr_p2p_step)
struct P2PPeers {
    double* mail[SGPR_MAX_RANKS];     // mailbox block of every rank, mapped on this device
};
struct P2PStep {
    P2PPeers peers;
    double* own_base;                 // this rank's two accumulation buffers (stride doubles apart)
    long long stride;
    double* F_d;
    uint8_t* owned_d;
};
int backward_grid(sgpr_context* h);
// training-time kernels of the step's environments (api.cu: sgpr_kernel_jacobian, sgpr_kernel_jacobian_batch):
// J [ncol, n_atoms, 3] += d Ke[b(j), m] / d x_j and W [B, ncol, 9] += sum_pairs r (x) dKe/dr, for the inducing LCEs sel
struct JacTarget {
    const int* sel;          // device [2 n_sel]: sorted inducing positions grouped by central species, then their columns
    int n_sel;
    int sel_first[SGPR_MAX_SPECIES + 1];   // host: range of each central species in sel
    int ncol;
    long long n_atoms;
    double* J;               // zeroed by the caller
    double* W;               // zeroed by the caller
    const double* cells;     // device [B, 9]
    const int* astr;         // device [N] structure of a cell-order atom; nullptr: one structure
};
int descriptor_jacobian_atoms(sgpr_context* h, const JacTarget& t, cudaStream_t st);
int unpack_descriptors(sgpr_context* h, long long rows, const double* packed_d, const int* src_row_d, double* full_d,
                       cudaStream_t st);

// ---- gemm.cu ----------------------------------------------------------------------
int gemm_energy_parts(int Ms);
int gemm_kernel_matrix(sgpr_context* h, double* Kmat, int ldk, const int* row_map_d, bool store_kc, cudaStream_t st,
                       const double* wmat = nullptr);
int gemm_covloss_parts(sgpr_context* h);
int gemm_covloss(sgpr_context* h, int64_t n_rows, cudaStream_t st);

// ---- i8gemm.cu --------------------------------------------------------------------
int i8_prepare_model(sgpr_context* h, bool weights_only);
int i8_prepare_covloss(sgpr_context* h);
int i8_ensure_step_buffers(sgpr_context* h, size_t n_rows, bool with_k8 = false);
int i8_energy_parts(int Ms);
int i8_kernel_matrix(sgpr_context* h, cudaStream_t st, bool store_k8 = false);
int i8_covloss_parts(sgpr_context* h);
int i8_covloss(sgpr_context* h, int64_t n_rows, cudaStream_t st);
int i8_back_projection(sgpr_context* h, cudaStream_t st);
int i8_setup_step(sgpr_context* h, cudaStream_t st);   // work lists of this step's GEMMs from row_first_d (one warp)
int gemm_back_projection(sgpr_context* h, cudaStream_t st);

// ---- api.cu: the prediction step as the MD driver runs it (single structure, no sharding) ---------------------------
bool md_warm_possible(sgpr_context* h, int64_t N, const int32_t* pbc_h, bool beta);
// graph = true: sgpr_predict's path (replays its own graph when warm); false: plain launches, for capture by the caller
int md_predict(sgpr_context* h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
               const int32_t* pbc_h, cudaStream_t st, double* E_d, double* F_d, double* W_d, double* beta_d, bool graph);

// ---- md.cu ----------------------------------------------------------------------------------------------------------
enum { kDriverMd = 1, kDriverRelax = 2 };
void drop_driver_graphs(sgpr_context* h);
// one step of a device driver: enqueue(true) runs it with plain launches (sizing steps, no graph); when warm, the step
// enqueued by enqueue(false) is captured once per key and replayed (key zero-filled before its fields are set: compared
// with memcmp)
int driver_graph_step(sgpr_context* h, const sgpr_context::DriverGraphKey& key, bool warm,
                      const std::function<int(bool)>& enqueue);
// an error met while enqueueing a driver step names the step: "<what> <state_d[0] + 1>: <message>"
int driver_name_step(sgpr_context* h, int rc, const long long* state_d, cudaStream_t st, const char* what);

}  // namespace sgpr
