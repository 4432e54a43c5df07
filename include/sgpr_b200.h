/* sgpr_b200.h -- C ABI of the B200-native SGPR prediction path (libsgpr_b200.so).
 *
 * Drop-in boundary for AutoForce's prediction hot path (SURVEY.md section 8b).  The
 * reference is pure Python (no FFI of its own); each entry point below names the
 * reference interface whose work it replaces (paths relative to the reference repo,
 * theforce v2021.09).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *   - plain C types only; every pointer is suffixed _h (host memory) or _d (device
 *     memory on the handle's CUDA device);
 *   - every function returns 0 on success, a negative sgpr_status on failure; the
 *     message of the last failure on the calling thread is sgpr_last_error();
 *   - never throws, never exits; one handle per CUDA device, not re-entrant;
 *   - all device work of a call is enqueued on the caller-supplied `stream`
 *     (a cudaStream_t passed as void*; NULL = the legacy default stream).  Calls that
 *     return host results synchronise that stream before returning;
 *   - float64 everywhere (the reference sets torch's default dtype to float64,
 *     theforce/__init__.py:13); atomic numbers are int32, indices int32/int64 as noted.
 */
#ifndef SGPR_B200_H
#define SGPR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGPR_ABI_VERSION 1
#define SGPR_MAX_SPECIES 8

typedef struct sgpr_context* sgpr_handle;

typedef enum {
    SGPR_OK = 0,
    SGPR_ERR_INVALID = -1,      /* bad argument / unsupported hyper-parameter        */
    SGPR_ERR_CUDA = -2,         /* CUDA runtime error (message has the details)      */
    SGPR_ERR_SPECIES = -3,      /* atomic number not in the handle's species table   */
    SGPR_ERR_GEOMETRY = -4,     /* singular cell / atom too far outside the cell     */
    SGPR_ERR_NOMEM = -5,
    SGPR_ERR_NO_DEVICE = -6,    /* no CUDA device: there is NO CPU fallback          */
    SGPR_ERR_RETRY = -7         /* an asynchronous step outgrew the buffers sized by an earlier
                                   step (sgpr_check): repeat it                       */
} sgpr_status;

/* Frozen model = kernel hyper-parameters + inducing set + weights.
 * Replaces what ActiveCalculator reads from PosteriorPotential on the hot path
 * (regression/gppotential.py:453-478, 548-649; SURVEY section 8 row a10):
 *   model.gp.kern.kernels[0].{exponent, cutoff, descriptor.{nmax, ylm.lmax, radii|unit,
 *   normalize}, _a},  model.X (LocalsData of Local: number, _r, _b),  model.mu,
 *   model.choli,  model.mean.weights/_weights,  model._vscale.
 * SeSoapKernel (similarity/sesoap.py:10-24, descriptor/sesoap.py:102-260) and
 * UniversalSoapKernel (similarity/universal.py:52-122, descriptor/soap.py:715-851) differ
 * only in the per-species length unit:  radii[s] = radii(Z_s)  resp.  = unit for all s.
 * All pointers are HOST pointers; the library copies what it needs. */
typedef struct {
    int32_t lmax;                 /* ylm.lmax,  <= 8                                  */
    int32_t nmax;                 /* radial order, nmax + 1 <= 12                     */
    double  xi;                   /* kernel exponent (universal.py:67,121)            */
    double  rc;                   /* cutoff of PolyCut(rc, n=2) (cutoff.py:33-44)     */
    int32_t normalize;            /* descriptor.normalize (sesoap.py:249-251)         */
    int32_t n_species;            /* size of the dense species table, <= 8            */
    int32_t species_Z[SGPR_MAX_SPECIES];     /* sorted atomic numbers; must cover every
                                     species of the inducing set AND of the structures */
    double  radii[SGPR_MAX_SPECIES];         /* length unit of neighbour species s     */
    int32_t central_enabled[SGPR_MAX_SPECIES]; /* 0 = species excluded as a centre
                                     (`a`/`a_not`, universal.py:44-49,85,101; the `a` of
                                     SubSeSoapKernel, similarity/sesoap.py:27-43)       */
    int32_t neighbor_enabled[SGPR_MAX_SPECIES]; /* 0 = neighbours of this species do not
                                     enter the descriptor (species outside the `b` list of
                                     SubSeSoap, descriptor/sesoap.py:263-335)            */
    int32_t M;                    /* number of inducing LCEs                          */
    const int64_t* ind_first_h;   /* [M+1] CSR offsets into ind_r / ind_b             */
    const double*  ind_r_h;       /* [nnz,3]  Local._r  (descriptor/atoms.py:36-52)   */
    const int32_t* ind_b_h;       /* [nnz]    Local._b  (atomic numbers)              */
    const int32_t* ind_Z_h;       /* [M]      Local.number                            */
    const double*  mu_h;          /* [M]      model.mu                                */
    const double*  mean_w_h;      /* [n_species] weights[Z]+_weights[Z]; 0 where the
                                     mean has no entry (gppotential.py:219-227)        */
    const double*  choli_h;       /* [M,M] row-major model.choli, or NULL             */
    const double*  vscale_h;      /* [n_species] model._vscale[Z] (inf where unseen,
                                     calculator/active.py:797-803), or NULL            */
    int32_t device;               /* CUDA device ordinal                              */
    double  lone_weight;          /* number of similarity kernels in model.gp.kern.kernels: each adds the
                                     lone-atoms term (similarity/similarity.py:41-43,94-103), so two
                                     neighbour-less LCEs of one species have k = lone_weight (1 for a single
                                     kernel, n for default_kernel(species=[...n...])); 0 is read as 1, a negative
                                     value switches the term off (secondary handles of a model that sums kernels
                                     with different hyper-parameters, INTEGRATION.md)                      */
} sgpr_model_desc;

/* ---- life cycle ------------------------------------------------------------------ */

/* Build a handle: uploads the model and evaluates the inducing descriptors Z_hat on the
 * device with the same kernels used for atoms.  Replaces the per-LCE cache
 * `kern.precalculate(loc)` -> loc.kern_0_value (similarity/universal.py:100-107). */
int sgpr_create(const sgpr_model_desc* desc, sgpr_handle* out);
void sgpr_destroy(sgpr_handle h);
const char* sgpr_last_error(void);
int sgpr_abi_version(void);

/* New weights after the reference's trainer refitted the model (make_munu,
 * regression/gppotential.py:548-601).  Any pointer may be NULL (= keep). */
int sgpr_set_weights(sgpr_handle h, const double* mu_h, const double* mean_w_h,
                     const double* choli_h, const double* vscale_h);

/* Append n_new inducing LCEs (CSR like sgpr_model_desc: ind_first_h [n_new+1], ind_r_h / ind_b_h indexed by
 * it) after the existing ones and replace the weights, whose sizes follow M: mu_h [M+n_new], choli_h
 * [(M+n_new)^2] or NULL (covloss unavailable until sgpr_set_weights provides one).  Replaces
 * PosteriorPotential.add_inducing (regression/gppotential.py:888-940) as driven by
 * ActiveCalculator.update_inducing (calculator/active.py:842-929).  On error the old model stays in place. */
int sgpr_append_inducing(sgpr_handle h, int32_t n_new, const int32_t* ind_Z_h, const int64_t* ind_first_h,
                         const double* ind_r_h, const int32_t* ind_b_h, const double* mu_h, const double* choli_h);

/* ---- the hot path ---------------------------------------------------------------- */

/* One ActiveCalculator.calculate() in prediction mode (calculator/active.py:425-611):
 * neighbour list (descriptor/atoms.py:348-363,402), descriptors (sesoap.py:161-260),
 * kernel vs the inducing set (similarity.py:17-43, universal.py:109-122),
 * E = sum(K mu) + mean (active.py:548-570), F = -dE/dxyz and the pair virial
 * (active.py:587-611).  Device-resident inputs and outputs.
 *   pos_d  [N,3]   positions (need not be wrapped into the cell)
 *   Z_d    [N]     atomic numbers
 *   cell_h [9]     row-major lattice vectors (zero rows allowed on non-periodic axes)
 *   pbc_h  [3]
 *   rank, world    atom sharding: this call evaluates the local energies of its share
 *                  of the atoms (contiguous range in the internal cell order) and the
 *                  forces on exactly those atoms; (0,1) = everything.
 *   E_d    [1]     sum of the owned atoms' local energies + the mean terms of the owned atoms
 *   F_d    [N,3]   forces on owned atoms, 0 elsewhere
 *   W_d    [9]     un-normalised pair virial sum_i r_ij (x) dE_i/dr_ij of owned
 *                  environments, index [a*3+b] = r_a g_b; stress = (W/V).flat[[0,4,8,5,2,1]]
 *   beta_d [N]     covloss (active.py:781-804) of owned atoms, or NULL to skip
 *   owned_d[N]     1 where this rank owns the atom (uint8), or NULL */
int sgpr_predict(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                 const double* cell_h, const int32_t* pbc_h, int32_t rank, int32_t world,
                 void* stream, double* E_d, double* F_d, double* W_d, double* beta_d,
                 uint8_t* owned_d);

/* Same with HOST buffers: what the calculator calls once per MD step.  Stages through
 * pinned memory; H2D of positions and D2H of E/F/W(/beta) are inside the call. */
int sgpr_predict_host(sgpr_handle h, int64_t N, const double* pos_h, const int32_t* Z_h,
                      const double* cell_h, const int32_t* pbc_h, int32_t rank, int32_t world,
                      double* E_h, double* F_h, double* W_h, double* beta_h, uint8_t* owned_h);

/* B independent structures under the handle's model in ONE call (calculator/active.py:425-611 once per structure):
 * testing a model on a trajectory, the images of an NEB, scoring a data set -- structures of tens to hundreds of atoms,
 * for which a call per structure is mostly fixed cost.
 *   first_h [B+1]   int64 host CSR offsets: structure b = atoms first_h[b] .. first_h[b+1]-1 (0-atom structures allowed)
 *   pos_d [Ntot,3], Z_d [Ntot]   device, structures concatenated (Ntot = first_h[B])
 *   cell_h [B,9], pbc_h [B,3]    host, per structure, same conventions as sgpr_predict
 *   E_d [B], W_d [B,9], F_d [Ntot,3], beta_d [Ntot] or NULL   device, caller's order
 * Per structure, E, W and beta mean exactly what they mean in sgpr_predict, and do not depend on the rest of the batch.
 * Errors: SGPR_ERR_INVALID for malformed first_h (not starting at 0, not monotone); SGPR_ERR_GEOMETRY / _SPECIES name
 * the first structure that failed in sgpr_last_error().  B = 0 does nothing.
 * Synchronises the stream once (sizing); never sharded; never replayed as a graph; leaves no state for
 * sgpr_kernel_backward.  sgpr_get_stats reports the batch's totals. */
int sgpr_predict_batch(sgpr_handle h, int32_t B, const int64_t* first_h, const double* pos_d, const int32_t* Z_d,
                       const double* cell_h, const int32_t* pbc_h, void* stream,
                       double* E_d, double* F_d, double* W_d, double* beta_d);

/* Atom-sharded prediction with a PEER-MEMORY force exchange over NVLink instead of the halo recompute
 * of sgpr_predict(rank, world): every rank evaluates only the environments it owns and accumulates all
 * pair forces in its own buffer; what it accumulated for atoms of other ranks (the halo) is then added
 * (red.global.add.f64, once per atom and component) into their owners' accumulation buffers through
 * the peer mappings.  Replaces the reference's all_reduce of the
 * [N,3] force array (calculator/active.py:601); the only collective left is the caller's all-reduce
 * of E_d[1] and W_d[9].
 *   peer_f_h [world]  host array of device pointers: peer_f_h[r] = rank r's accumulation buffer
 *                     (3*N doubles, cell order, zero on entry; entries of atoms the rank does not own hold scratch afterwards), mapped into this device's address space
 *                     (e.g. torch symmetric memory / cudaIpcOpenMemHandle); peer_f_h[rank] is local.
 * After ALL ranks have finished this call (the caller's E/W all-reduce is the barrier), each rank reads
 * its own forces with sgpr_p2p_collect. */
int sgpr_predict_p2p(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                     const double* cell_h, const int32_t* pbc_h, int32_t rank, int32_t world,
                     void* stream, const uint64_t* peer_f_h, double* E_d, double* W_d);
/* own accumulation buffer -> F_d [N,3] (caller's atom order; 0 for atoms of other ranks), owned_d [N]. */
int sgpr_p2p_collect(sgpr_handle h, void* stream, const double* own_f_d, double* F_d, uint8_t* owned_d);

/* The whole exchange step in ONE call and without any collective library: sgpr_predict_p2p + the all-reduce of E and the
 * 3x3 virial (calculator/active.py:562,602) + sgpr_p2p_collect.  Every rank owns one symmetric block of peer-mapped
 * memory (zero-initialised, e.g. torch symmetric memory), laid out in doubles as
 *     [2][3N + 8]      force accumulation buffers (cell order); steps alternate between them
 *     [2][world][16]   mailboxes: slot r of one half = rank r's {E, W[9]} and a 64-bit step stamp at [15]
 * (which half a step uses is the low bit of a step counter that lives on the device: the arguments of a warm step are
 * identical from step to step, so it replays as ONE CUDA graph)
 * peer_base_h[r] = base address of rank r's block as mapped on THIS device.  Per step each rank
 *   1. clears its accumulation buffer of the next step,  2. evaluates the environments it owns and pushes the forces it
 *   accumulated on atoms of other ranks into their buffers over NVLink,  3. writes its E and virial into EVERY rank's mailbox and then
 *   the stamp (st.release.sys),  4. waits until all stamps of the step have arrived in its own mailbox -- every
 *   rank's push has then finished -- and sums the world contributions in rank order (bit-identical on all
 *   ranks),  5. copies its own forces to F_d [N,3] (caller's order, rows of owned atoms) and fills owned_d [N].
 * E_d [1], W_d [9], F_d, owned_d are device pointers; everything is enqueued on `stream` (warm steps: one CUDA graph,
 * no host synchronisation -- see "Asynchronous steps").  All ranks must call it once per step, the same number of times.
 * A peer that never arrives is given up after 10 s (reported by sgpr_check); the GPU is never left spinning. */
int sgpr_p2p_step(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                  const int32_t* pbc_h, int32_t rank, int32_t world, void* stream, const uint64_t* peer_base_h,
                  double* E_d, double* F_d, double* W_d, uint8_t* owned_d);

/* Kernel matrix cov = model.gp.kern(atoms, model.X)  (calculator/active.py:464,
 * regression/gppotential.py:47-50,63-64; similarity/similarity.py:17-31).
 *   K_d [N,M] row-major, atoms and inducing LCEs in the caller's order. */
int sgpr_kernel_forward(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                        const double* cell_h, const int32_t* pbc_h, void* stream, double* K_d);

/* Vector-Jacobian product of the last sgpr_kernel_forward: given gK = dL/dcov [N,M]
 * returns dL/dxyz [N,3] and dL/dcell [9] -- what torch.autograd.grad(E, xyz / lll) does
 * in the reference (calculator/active.py:587-599, gppotential.py:905-911). */
int sgpr_kernel_backward(sgpr_handle h, const double* gK_d, void* stream, double* gpos_d,
                         double* gcell_h);

/* Training-time kernels of the structure of the LAST sgpr_kernel_forward against the inducing LCEs
 * m0 <= m < m1 (caller's order), i.e. what EnergyForceKernel.forces_energy / virial_energy
 * (regression/gppotential.py:66-77) build from SimilarityKernel "leftgrad" / "virial"
 * (similarity/universal.py:124-183):
 *   J_d [(m1-m0), N, 3] = d (sum_i K[i,m]) / d xyz       (leftgrad; forces_energy = -J)
 *   W_d [(m1-m0), 9]    = sum_pairs r (x) dK/dr, row-major 3x3, NOT divided by the volume
 *                         (virial_energy = W.flat[[0,4,8,5,2,1]])
 * These are the true derivatives (they agree with torch.autograd through the reference's forward pass);
 * the reference's hand-written leftgrad drops contributions when an atom occurs twice in one environment
 * (index assignment g[j] += f, universal.py:148) -- see tests/golden/make_golden_train.py.
 * All m0 <= m < m1 are evaluated by one launch of the Jacobian kernel (as in sgpr_kernel_jacobian_batch); J_d and
 * W_d agree with it to rounding (atomic accumulation). */
int sgpr_kernel_jacobian(sgpr_handle h, int32_t m0, int32_t m1, void* stream, double* J_d, double* W_d);

/* Training-time kernels of B independent structures in one call: for every data structure b and every inducing LCE
 * m0 <= m < m1 the energy_energy, forces_energy and virial_energy blocks that make_munu stacks
 * (regression/gppotential.py:63-77 EnergyForceKernel(first=[...]), 548-601 make_munu; update_data / update_inducing).
 * Replaces one sgpr_kernel_forward + sgpr_kernel_jacobian pair per structure.
 *   first_h [B+1], pos_d, Z_d, cell_h [B,9], pbc_h [B,3]   as in sgpr_predict_batch (0-atom structures, own cells, mixed pbc)
 *   Ke_d [B, m1-m0]          sum_{i in b} K[i,m], lone-lone term included (K.sum(0) of sgpr_kernel_forward per
 *                            structure); fixed summation order: bit-identical whatever else is in the batch
 *   J_d  [m1-m0, Ntot, 3]    d Ke[b(j), m] / d x_j, caller's atom order, layout and sign of sgpr_kernel_jacobian
 *   W_d  [B, m1-m0, 9]       sum_pairs r (x) dK/dr per structure, NOT divided by the volume (sgpr_kernel_jacobian's W_d)
 * J_d and W_d both NULL: Ke only (no Jacobian stage); only one of them NULL is SGPR_ERR_INVALID.  J and W are
 * accumulated with red.global.add.f64 and agree with a call on the structure alone to rounding.
 * Errors: SGPR_ERR_INVALID for malformed first_h or m0 < 0, m1 > M, m0 > m1; SGPR_ERR_GEOMETRY / _SPECIES name the first
 * structure that failed in sgpr_last_error().  B = 0 does nothing.
 * Synchronises the stream once (sizing); never sharded; never replayed as a graph; leaves no state for
 * sgpr_kernel_backward / sgpr_kernel_jacobian (the next single-structure step sizes again).  sgpr_get_stats reports the
 * batch's totals. */
int sgpr_kernel_jacobian_batch(sgpr_handle h, int32_t B, const int64_t* first_h, const double* pos_d, const int32_t* Z_d,
                               const double* cell_h, const int32_t* pbc_h, int32_t m0, int32_t m1, void* stream,
                               double* Ke_d, double* J_d, double* W_d);

/* ---- parity hooks (used by tests; same kernels as the hot path) --------------------- */

/* Neighbour list as ASE's NeighborList(N*[rc/2], skin=0, self_interaction=False,
 * bothways=True) returns it through get_neighbors(a) (descriptor/atoms.py:348-366):
 * CSR over atoms in the caller's order, offsets relative to the given positions.
 *   first_d [N+1] int64;  j_d [capacity] int32;  S_d [capacity,3] int8
 *   *nnz_h receives the number of pairs; if it exceeds `capacity` nothing is written to
 *   j_d/S_d and the call still returns SGPR_OK (call again with a larger buffer). */
int sgpr_neighbors(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                   const double* cell_h, const int32_t* pbc_h, void* stream,
                   int64_t* first_d, int32_t* j_d, int8_t* S_d, int64_t capacity, int64_t* nnz_h);

/* Normalised descriptors of all atoms in the reference's dense block layout
 * p[s1,s2,n1,n2,l] (descriptor/sesoap.py:195-203,248-258; block [s1,s2] <-> sparse
 * index (Z_s2, Z_s1)):  P_d [N, S*S*(nmax+1)^2*(lmax+1)]. */
int sgpr_descriptors(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d,
                     const double* cell_h, const int32_t* pbc_h, void* stream, double* P_d);

/* Same layout for the inducing LCEs (loc.kern_0_value): Zhat_d [M, S*S*(nmax+1)^2*(lmax+1)]. */
int sgpr_inducing_descriptors(sgpr_handle h, void* stream, double* Zhat_d);

/* Asynchronous steps.  The first sgpr_predict / sgpr_predict_p2p / sgpr_predict_host of a given shape (atom count,
 * rank, world) is a SIZING step: it synchronises the stream once to learn the pair count and the per-species row
 * ranges.  Later steps of the same shape need neither: both stay on the device (capacity + overflow flag, work lists of
 * the GEMMs written by a one-warp kernel), so the host enqueues the whole step without waiting -- the same launch
 * sequence every step.
 *   - sgpr_predict_host always does this and validates the step itself (an overflowing step is repeated as a sizing
 *     step inside the same call);
 *   - the device-pointer entry points do it only after sgpr_set_async(h, 1), because they return before the step has
 *     run: call sgpr_check(h, &n_pairs) after synchronising the stream -- SGPR_OK, or SGPR_ERR_RETRY / _SPECIES /
 *     _GEOMETRY if any step since the last check was invalid (its outputs are then meaningless; an invalid step never
 *     writes outside its buffers).
 * Non-periodic cells, halo-recompute sharding (sgpr_predict with world > 1) and the FP64 DMMA path always size. */
int sgpr_set_async(sgpr_handle h, int32_t on);
int sgpr_check(sgpr_handle h, int64_t* n_pairs_out);

/* ---- molecular dynamics on the device ------------------------------------------------
 * What ASE's VelocityVerlet / Langevin do around ActiveCalculator in prediction mode (calculator/active.py:425-611,
 * covloss 492-499), with positions, momenta and forces resident on the device.  Units are the caller's (ASE: eV, A, amu,
 * ASE time); pos_d and mom_d stay unwrapped, as in ASE.
 *   NVE (langevin = 0), ASE's operation order:   p += dt/2 F;  r += dt p/m;  F = F(r);  p += dt/2 F
 *   NVT (langevin = 1), BAOAB:  p += dt/2 F;  r += dt/2 p/m;  p = c1 p + c2 sqrt(m kT) xi;  r += dt/2 p/m;  F = F(r);
 *                               p += dt/2 F    with c1 = exp(-friction dt), c2 = sqrt(1 - c1^2), no centre-of-mass fix;
 *                               xi = Philox4x32-10 normals keyed by seed and counted by (atom, step): sgpr_math.cuh
 * Device state state_d [4] int64: 0 steps done (the global step, also the noise counter of the next step), 1 the step
 * at which max(beta) > ediff first held (0 = the starting structure; -1 = none), 2 = 1 when the step state_d[0]+1 was
 * not integrated because its prediction was invalid, 3 the step at which the current sgpr_md_steps call began.
 * Once state_d[1] >= 0 or state_d[2] = 1 every later step leaves positions, momenta, forces and beta unchanged. */
typedef struct {
    double   dt;                  /* time step                                                       */
    double   friction;            /* Langevin friction (1/time); unused for NVE                        */
    double   kT;                  /* Langevin temperature (energy); unused for NVE                     */
    double   ediff;               /* stop when max(beta) > ediff (the comparison of prediction mode: NaN does not
                                     stop, inf does)                                                    */
    uint64_t seed;                /* Philox key of the Langevin noise                                  */
    int32_t  langevin;            /* 0 = velocity Verlet, 1 = BAOAB Langevin                           */
    int32_t  stop_on_uncertain;   /* 1: evaluate covloss every step (beta_d required) and stop          */
} sgpr_md_params;

/* Start of a run: F_d [N,3] (and beta_d [N] if p->stop_on_uncertain) = forces (covloss) of pos_d, state_d = {0, -1 or 0, 0,
 * 0}.  Enqueued on `stream` like sgpr_predict in asynchronous mode: after synchronising, sgpr_check reports an invalid
 * evaluation (SGPR_ERR_RETRY: call sgpr_md_init again). */
int sgpr_md_init(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const double* cell_h,
                 const int32_t* pbc_h, const sgpr_md_params* p, void* stream, double* F_d, double* beta_d,
                 int64_t* state_d);

/* Enqueue n_steps MD steps.  pos_d, mom_d [N,3] and F_d (forces of pos_d on entry) are updated in place; mass_d [N];
 * thermo_d [n_steps, 11] receives one row per step done by this call, {E_pot, E_kin, W[9]} (W as in sgpr_predict; E_kin
 * = sum p^2/2m in a fixed order); beta_d [N] (or NULL without stop_on_uncertain) the covloss of the current positions.
 * Warm steps (periodic cell, buffers sized by an earlier step of the same shape) need no host synchronisation: a step is
 * one CUDA graph launch.  After synchronising the stream, read state_d and call sgpr_check: SGPR_ERR_RETRY means a step
 * outgrew the buffers and was NOT integrated (state_d[2] = 1): enqueue the remaining steps again; they size first.
 * Other errors (an atom more than 120 cells outside the cell, unknown species) also leave the state of the last good
 * step.  Errors found while enqueueing (sizing steps: non-periodic cells size on every step) name the step. */
int sgpr_md_steps(sgpr_handle h, int64_t N, double* pos_d, double* mom_d, const int32_t* Z_d, const double* mass_d,
                  const double* cell_h, const int32_t* pbc_h, const sgpr_md_params* p, int32_t n_steps, void* stream,
                  double* F_d, double* thermo_d, double* beta_d, int64_t* state_d);

/* ---- geometry relaxation on the device ------------------------------------------------
 * ASE's FIRE optimiser (ase/optimize/fire.py of ASE 3.22-3.23, downhill_check=False) around the prediction step, with
 * positions, velocities and forces resident on the device.  Iteration k, with the forces F of the positions r known:
 *   converged <=> max_i |F_i|^2 < fmax^2   (tested before every step, the starting structure included)
 *   first step: v = 0;  later: if F.v > 0:  v = (1-a) v + a |v| F/|F|;  if Nsteps > Nmin: dt = min(dt finc, dtmax),
 *                                          a *= fa;  Nsteps += 1
 *                               else:     v *= 0;  a = astart;  dt *= fdec;  Nsteps = 0
 *   v += dt F;  dr = dt v;  if |dr| > maxstep: dr *= maxstep/|dr| (norm over all atoms);  r += dr;  F = F(r)
 * fixed_d (uint8 [N], or NULL): the forces of atoms with fixed_d[i] != 0 are zero in every use above (ASE's FixAtoms
 * through get_forces()), so they never move; energy and virial are those of all atoms.
 * fire_d [6] double: {dt, a, F.v, F.F, v.v, max_i |F_i|^2} -- the FIRE scalars and the reductions of the current F, v.
 * state_d [6] int64: 0 steps done, 1 the step at which max(beta) > ediff first held (-1 = none), 2 = 1 when the step
 * state_d[0]+1 was not done because its prediction was invalid, 3 the step at which the current sgpr_relax_steps call
 * began, 4 the step whose forces met fmax (-1 = none), 5 FIRE's Nsteps.  Once state_d[1] >= 0, state_d[2] = 1 or
 * state_d[4] >= 0 every later step leaves positions, velocities, forces, beta and fire_d unchanged. */
typedef struct {
    double   dt;                  /* FIRE (ASE's names and defaults): initial time step, 0.1                */
    double   maxstep;             /* largest |dr| of a step (norm over all atoms), 0.2                       */
    double   dtmax;               /* 1.0                                                                   */
    double   finc, fdec;          /* 1.1, 0.5                                                              */
    double   astart, fa, a;       /* 0.1, 0.99, 0.1 (a: initial mixing)                                    */
    double   fmax;                /* convergence: max_i |F_i| < fmax                                        */
    double   ediff;               /* stop when max(beta) > ediff (as sgpr_md_params)                        */
    int32_t  Nmin;                /* 5                                                                     */
    int32_t  stop_on_uncertain;   /* 1: evaluate covloss every step (beta_d required) and stop               */
} sgpr_relax_params;

/* Start of a relaxation: F_d [N,3] (and beta_d [N] if p->stop_on_uncertain) of pos_d, fixed rows zeroed; fire_d = {p->dt,
 * p->a, ...}; state_d = {0, -1 or 0, 0, 0, 0 if the start meets p->fmax else -1, 0}.  Enqueued on `stream`; after
 * synchronising, sgpr_check reports an invalid evaluation (SGPR_ERR_RETRY: call sgpr_relax_init again). */
int sgpr_relax_init(sgpr_handle h, int64_t N, const double* pos_d, const int32_t* Z_d, const uint8_t* fixed_d,
                    const double* cell_h, const int32_t* pbc_h, const sgpr_relax_params* p, void* stream, double* F_d,
                    double* beta_d, double* fire_d, int64_t* state_d);

/* Enqueue n_steps FIRE steps.  pos_d, vel_d [N,3], F_d (forces of pos_d on entry), beta_d, fire_d and state_d are
 * updated in place.  The call first re-tests the current forces against p->fmax (state_d[4]), as ASE's run(fmax) does.
 * trace_d [n_steps, 13] receives one row per step done by this call: {E_pot, max_i |F_i|, dt, a, W[9]} (dt and a after
 * the step's update).  Warm steps replay one CUDA graph each; the overflow protocol and the errors are sgpr_md_steps':
 * SGPR_ERR_RETRY with state_d[2] = 1 means the step was not done: enqueue the remaining steps again. */
int sgpr_relax_steps(sgpr_handle h, int64_t N, double* pos_d, double* vel_d, const int32_t* Z_d, const uint8_t* fixed_d,
                     const double* cell_h, const int32_t* pbc_h, const sgpr_relax_params* p, int32_t n_steps,
                     void* stream, double* F_d, double* trace_d, double* beta_d, double* fire_d, int64_t* state_d);

/* Explicit local chemical environments (reference `Local` objects: number, _r, _b; descriptor/atoms.py:36-52) against
 * the inducing set -- the similarity interface on LCEs rather than structures:
 *   K_d [n_env, M]   = kern(locs, X)            (similarity/similarity.py:17-43, universal.py:109-122 incl. the
 *                                                 lone-atoms term), columns in the caller's inducing order; with the
 *                                                 handle's own LCEs as input this is the M x M matrix of
 *                                                 regression/gppotential.py:511 / 781.
 *   P_d [n_env, S*S*(nmax+1)^2*(lmax+1)] = kern.call_descriptor(loc, grad=False) / precalculate (universal.py:97-107)
 *                                                 in the dense block layout of sgpr_descriptors.
 * Environments are host CSR arrays like sgpr_model_desc.ind_*; either output may be NULL.  Synchronises the stream. */
int sgpr_kernel_envs(sgpr_handle h, int32_t n_env, const int32_t* env_Z_h, const int64_t* env_first_h,
                     const double* env_r_h, const int32_t* env_b_h, void* stream, double* K_d, double* P_d);

/* ---- introspection ------------------------------------------------------------------ */

typedef struct {
    int64_t n_atoms;          /* atoms of the last call                                */
    int64_t n_active;         /* environments evaluated (owned + halo)                 */
    int64_t n_pairs;          /* neighbour pairs of the evaluated environments         */
    int32_t d_packed;         /* packed descriptor length used by the GEMMs            */
    int32_t d_full;           /* S*S*(nmax+1)^2*(lmax+1)                               */
    int64_t kernel_launches;  /* CUDA kernels launched by the last hot-path call        */
    double  gemm_flops;       /* flops executed by the two kernel GEMMs, last call     */
    double  covloss_flops;    /* flops executed by the covloss GEMM, last call         */
    double  i8_ops;           /* int8 tensor-core operations of the sliced GEMMs (0 on the
                                 FP64 DMMA path), last call                            */
    float   ms_nl, ms_desc, ms_gemm, ms_force, ms_beta, ms_total; /* device time per stage
                                 of the last call (CUDA events), valid if timing is on */
} sgpr_stats;

int sgpr_get_stats(sgpr_handle h, sgpr_stats* out);
int sgpr_enable_timing(sgpr_handle h, int32_t on);

#ifdef __cplusplus
}
#endif
#endif /* SGPR_B200_H */
