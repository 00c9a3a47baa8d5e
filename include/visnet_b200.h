/* visnet_b200.h -- C ABI of the B200-native ViSNet energy/force engine.
 *
 * Drop-in boundary for the one hot path of microsoft/AI2BMD: the per-MD-step ViSNet evaluation over a
 * packed batch of protein fragments.  Each entry point names the reference interface it replaces
 * (paths relative to the reference tree).  Plain pointers and sizes only -- no torch types.  Every
 * function returns 0 on success or a negative vb_status; the message is available from vb_last_error().
 * There is no CPU fallback: every compute entry fails with VB_ERR_CUDA when no sm_100 device is usable.
 *
 * Units/dtypes are the reference's: positions in Angstrom, energies in eV, forces in eV/Angstrom, fp32.
 */
#ifndef VISNET_B200_H
#define VISNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vb_handle vb_handle;

typedef enum {
    VB_OK = 0,
    VB_ERR_ARG = -1,      /* bad argument / hyper-parameter mismatch */
    VB_ERR_CUDA = -2,     /* CUDA runtime error (no device, launch failure, ...) */
    VB_ERR_STATE = -3,    /* call order (e.g. forward before set_topology) */
    VB_ERR_ALLOC = -4
} vb_status;

/* Hyper-parameters of the checkpoint (src/ViSNet/model/visnet.py:14-30; both shipped checkpoints:
 * embedding_dimension 128, num_layers 6, num_heads 8, num_rbf 32, lmax 1, cutoff 5.0,
 * max_num_neighbors 32).  The kernels are specialised for exactly these; vb_create() rejects others. */
typedef struct {
    int32_t hidden_channels;
    int32_t num_layers;
    int32_t num_heads;
    int32_t num_rbf;
    int32_t max_num_neighbors;
    float cutoff;
} vb_hparams;

/* Order and element counts ("name:count;...") of the flat fp32 weight blob vb_create() expects.
 * Replaces: ViSNet.load_state_dict in load_model(), src/ViSNet/model/visnet.py:73-93. */
const char* vb_weight_manifest(void);

/* Create an engine on CUDA device `device` from a host weight blob laid out per vb_weight_manifest().
 * Replaces: get_visnet_model(model_path, device) / ViSNetModel.__init__,
 *           src/Calculators/visnet_calculator.py:36-45,184-204. */
int vb_create(const float* weights_host, size_t n_floats, const vb_hparams* hp, int device, vb_handle** out);
void vb_destroy(vb_handle* h);
const char* vb_last_error(const vb_handle* h);   /* h may be NULL: last creation error */

/* Static topology of the packed batch: atomic numbers and graph ids (sorted, contiguous) of N atoms in
 * G fragments -- host pointers, copied.  max_edges <= 0 selects the worst case N*32 (always safe); a smaller value
 * trims the workspace and is a promise by the caller that no step produces more directed edges (incl. self-loops):
 * vb_forward_host verifies it after the fact and fails, the asynchronous entry points cannot.
 * Replaces: the z / batch members of FragmentData (src/AIMD/fragment.py:7-13) that
 *           ViSNetModel.collate() uploads every step (visnet_calculator.py:47-52). */
int vb_set_topology(vb_handle* h, int64_t n_atoms, int64_t n_graphs, const int64_t* z_host,
                    const int64_t* batch_host, int64_t max_edges);

/* One evaluation, device buffers, asynchronous on `stream` (a cudaStream_t passed as void*).
 *   pos_dev[N*3] -> energy_dev[G], forces_dev[N*3].
 * Replaces: ViSNet.forward, src/ViSNet/model/visnet.py:135-166 (energy + autograd force). */
int vb_forward(vb_handle* h, const float* pos_dev, float* energy_dev, float* forces_dev, void* stream);

/* One evaluation with HOST buffers (pinned staging + H2D/D2H inside), synchronous.
 * Replaces: ViSNetModel.dl_potential_loader(FragmentData) -> (e[G,1], f[N,3]),
 *           src/Calculators/visnet_calculator.py:54-63. */
int vb_forward_host(vb_handle* h, const float* pos_host, float* energy_host, float* forces_host);

/* Whole-protein reduction map: F_prot[dst_atom[m]] += sign[m] * F[src_atom[m]], E_prot = sum_g frag_sign[g]*E_g.
 * Replaces: DipeptideBondedCombiner.energy_combine / forces_combine, src/Calculators/combiner.py:11-41
 *           (select_index / origin_index built at src/Fragmentation/distancefrag.py:335-353) and the
 *           dipeptide / ACE-NME split of src/Calculators/bonded.py:91-93. */
int vb_set_protein_map(vb_handle* h, int64_t n_protein_atoms, int64_t n_map, const int32_t* src_atom_host,
                       const int32_t* dst_atom_host, const float* sign_host, const float* frag_sign_host);

/* Evaluation + signed scatter into ef_prot_dev[3*n_protein_atoms + 1] (forces, then the energy in the last
 * slot); the buffer is overwritten.  With several GPUs each rank calls this on its shard of fragments and
 * the caller all-reduces ef_prot_dev (NCCL sum).  Replaces: DLBondedCalculator.__call__, bonded.py:102-123. */
int vb_forward_protein(vb_handle* h, const float* pos_dev, float* ef_prot_dev, void* stream);

/* ---- Device-resident MD step (SURVEY section 8f, rank 3 and the first half of rank 1) ------------------------
 * State (protein positions / velocities, fp64) stays on the GPU; one step is
 *   kick1 (half-kick + drift) -> eval (place fragment atoms, ViSNet, signed reduction into ef [+ non-bonded term]
 *   [+ restraints]) -> kick2.
 * Replaces: the ASE Langevin loop the reference runs (src/AIMD/simulator.py:96-137: Langevin(dt = 1 fs, 300 K,
 *           friction 0.001/fs), MaxwellBoltzmannDistribution start; ASE 3.22 ase/md/langevin.py step()) and the
 *           per-step fragment coordinate rebuild with cap hydrogens on the acceptor->removed ray
 *           (src/Fragmentation/distancefrag.py:34-54), without the Amber-term LBFGS refinement.
 * Units as ASE: eV, Angstrom, amu; dt in Angstrom*sqrt(amu/eV), friction in 1/that; kT in eV.  friction = 0 is
 * velocity Verlet (no random numbers, no centre-of-mass correction).  Normals come from Philox4x32-10 keyed by
 * (seed; step, component): every rank of a sharded run draws the same numbers.
 *
 * vb_md_setup: recipe per FRAGMENT atom a (arrays of length N): real[a] = protein index, or -1 for an added
 * hydrogen placed at P[acc[a]] + unit(P[rem[a]] - P[acc[a]]) * blen[a].  ef_prot_dev[3*n_protein + 1] is the
 * caller-owned force/energy buffer (must hold forces of the current positions before the first kick1: call
 * vb_md_eval after vb_md_set_state).  Requires vb_set_protein_map with the same n_protein_atoms. */
int vb_md_setup(vb_handle* h, int64_t n_protein_atoms, const double* masses_host, const int32_t* real_host,
                const int32_t* acc_host, const int32_t* rem_host, const float* blen_host, double dt, double kT,
                double friction, uint64_t seed, float* ef_prot_dev);
/* Optional externally supplied normals, device array [pool_steps][2][3*n_protein] (xi, eta), step s reads row
 * s % pool_steps; (NULL, 0) returns to Philox.  For parity tests against a host integrator. */
int vb_md_set_normals(vb_handle* h, const double* pool_dev, int64_t pool_steps);
int vb_md_set_state(vb_handle* h, const double* x_host, const double* v_host, int64_t step);
/* The three phases, asynchronous on `stream`.  With several GPUs every rank holds the whole-protein state and its
 * own shard of fragments: kick1; eval; all-reduce ef_prot_dev (NCCL sum, by the caller); kick2. */
int vb_md_kick1(vb_handle* h, void* stream);
int vb_md_eval(vb_handle* h, void* stream);
int vb_md_kick2(vb_handle* h, void* stream);
/* Single GPU: n_steps whole steps, each one replay of a captured CUDA graph, no host synchronisation. */
int vb_md_run(vb_handle* h, int64_t n_steps, void* stream);
/* Synchronises; any of x_host / v_host / step_out may be NULL.  epot_hist_host[n_hist] receives the potential
 * energies recorded at the end of the last n_hist steps (oldest first). */
int vb_md_get_state(vb_handle* h, double* x_host, double* v_host, int64_t* step_out, double* epot_hist_host,
                    int64_t n_hist);

/* ---- Non-bonded MM term (SURVEY section 8f, rank 2) ---------------------------------------------------------------
 * All ordered pairs (src j, dst i), j != i, except pairs listed in the exclusion table (atoms sharing a dipeptide,
 * src/Fragmentation/distancefrag.py:355-363; pair list src/AIMD/protein.py:133-151): Lennard-Jones with
 * sigma_ij = (sigma_i + sigma_j)/2 [nm], eps_ij = sqrt(eps_i eps_j) [kJ/mol], plus Coulomb; forces summed on dst,
 * energy halved; results in eV and eV/Angstrom.  Replaces: MMNonBondedCalculator.set_parameters / __call__,
 * src/Calculators/nonbonded.py:24-63.  The exclusion table is CSR over protein atoms, each row strictly ascending.
 * [atom_lo, atom_hi) are the destination atoms this handle computes (a sharded run gives every rank a slice and
 * all-reduces the buffer). */
int vb_set_nonbonded(vb_handle* h, int64_t n_protein_atoms, const float* charges_host, const float* sigmas_nm_host,
                     const float* epsilons_kj_host, const int32_t* excl_rowptr_host, const int32_t* excl_col_host,
                     int64_t atom_lo, int64_t atom_hi);
/* ef_prot_dev[3*n + 1] += non-bonded forces / energy at prot_pos_dev[n*3] (fp32 positions as the reference casts
 * them, nonbonded.py:39).  Accumulates: zero the buffer for the bare term, or call after vb_forward_protein for
 * bonded + non-bonded (FragmentCalculator.calculate, src/Calculators/fragment.py:50-68).  Once set, vb_md_eval
 * adds the term too. */
int vb_nonbonded(vb_handle* h, const float* prot_pos_dev, float* ef_prot_dev, void* stream);

/* ---- Hookean restraints (pre-equilibration and hydrogen-bond constraints) ------------------------------------------
 * point (a, p0, k, rt): d = p0 - x_a, r = |d|; if r > rt: F_a += k (r - rt) d/r, E += k (r - rt)^2 / 2.
 * pair (i, j, k, rt):   d = x_j - x_i, r = |d|; if r > rt: F_i += k (r - rt) d/r, F_j -= k (r - rt) d/r, E += same.
 * k in eV/Angstrom^2, rt and anchors in Angstrom; no periodic images.  Anchors are fixed copies, they do not follow the
 * atom.  [atom_lo, atom_hi) are the destination atoms this handle computes (a sharded run gives every rank a slice and
 * all-reduces the buffer); a restraint's energy is counted where its first atom is computed.
 * Replaces: ASE 3.22 ase/constraints.py Hookean (adjust_forces / adjust_potential_energy) as the reference uses it:
 *           position restraints of the pre-equilibration (src/AIMD/simulator.py:139-166) and the hydrogen-bond springs
 *           of --constraints (simulator.py:168-180, pairs from PDBAnalyzer.find_bonded_atoms, src/utils/utils.py:169-221).
 *           Host helpers that build the sets: ai2bmd_b200/restraints.py. */
typedef struct {
    int64_t n_point; const int32_t* point_atom; const double* point_anchor /*[n][3]*/; const double* point_k; const double* point_rt;
    int64_t n_pair;  const int32_t* pair_ij /*[n][2]*/; const double* pair_k; const double* pair_rt;
    int64_t atom_lo, atom_hi;
} vb_restraint_set;
/* Host pointers, copied.  Requires vb_set_protein_map (which drops the set again).  Both counts 0 removes the term.
 * VB_ERR_ARG for an atom index outside [0, n_protein), i == j in a pair, a negative or non-finite k or rt, a non-finite
 * anchor or a bad slice.  Synchronises the device before it replaces the arrays; captured graphs are dropped.  Once set,
 * vb_md_eval / vb_md_run add the term after the bonded and non-bonded terms (before the automatic all-reduce). */
int vb_set_restraints(vb_handle* h, const vb_restraint_set* rs);
/* ef_prot_dev[3*n + 1] += restraint forces / energy at prot_pos_dev[n*3] (fp64 positions); adds nothing while no
 * restraints are set.  Two calls on the same input give bit-identical results (no atomics). */
int vb_restraints(vb_handle* h, const double* prot_pos_dev, float* ef_prot_dev, void* stream);

/* ---- Per-step refinement of the added (cap) hydrogens (SURVEY section 8f, rank 1) -----------------------------------
 * One LBFGS call (lr, max_iter, tolerance_grad, tolerance_change; no line search, fresh state) on the Amber energy of all
 * dipeptides, moving only the added hydrogens -- what the reference runs every MD step between placing them and the
 * ViSNet evaluation.  The problem is given as flat term arrays whose atom indices address the PACKED FRAGMENT position
 * buffer [N][3] of vb_set_topology: every term that contains an optimised hydrogen, with its own parameters (Amber
 * units: kcal/mol, Angstrom, radians; qq = product of prmtop charges).  mirror_dst/mirror_src: fragment atoms that are
 * copies of relaxed ones (the ACE-NME fragments take their hydrogens from the neighbouring dipeptides,
 * src/Fragmentation/distancefrag.py:286-307) and are re-copied after the relaxation.
 * Replaces: HydrogenOptimizer.optimize_hydrogen + the five energy terms, src/Fragmentation/hydrogen/energies.py:9-60,
 *           211-242 (tables: hydrogen/ctable.py:58-240), called from DistanceFragment.get_fragments,
 *           src/Fragmentation/distancefrag.py:56-92.  Host helper that builds the arrays from prmtop tables:
 *           ai2bmd_b200/caph.py.  Once set, vb_md_eval / vb_md_run refine after placing the fragment atoms. */
typedef struct {
    int64_t n_h;      const int32_t* h_idx;                                              /* optimised hydrogens        */
    int64_t n_bonds;  const int32_t* bond_ij;   const float* bond_k;  const float* bond_r0;      /* [n][2]             */
    int64_t n_angles; const int32_t* angle_ijk; const float* angle_k; const float* angle_t0;     /* [n][3]             */
    int64_t n_dih;    const int32_t* dih_ijkl;  const float* dih_k;   const float* dih_n; const float* dih_p;  /* [n][4] */
    int64_t n_pairs;  const int32_t* pair_ij;   const float* pair_a;  const float* pair_b; const float* pair_qq;
    int64_t n_mirror; const int32_t* mirror_dst; const int32_t* mirror_src;
    float scnb, scee;                 /* 1-4 scaling of the reference's HydrogenOptimizer: 1.2, 2.0                  */
    int32_t max_iter;                 /* 10 in the reference                                                         */
    float lr, tol_grad, tol_change;   /* 0.1, 0.1, 0.01 in the reference                                             */
} vb_caph_problem;
int vb_set_caph(vb_handle* h, const vb_caph_problem* problem);          /* host pointers, copied */
/* Refine a packed fragment position buffer in place (device pointer), asynchronous on `stream`. */
int vb_caph_relax(vb_handle* h, float* pos_dev, void* stream);

/* ---- One-shot all-reduce over NVLink peer memory (SURVEY section 8e) ---------------------------------------------
 * One process per GPU.  vb_comm_init allocates this rank's window (2 parities x world slots of max_floats) and returns
 * its 64-byte CUDA IPC handle; the caller exchanges the handles of all ranks (any host transport: torch.distributed,
 * MPI, a file) and passes them, in rank order, to vb_comm_connect.  From then on every evaluation that produces the
 * whole-protein buffer (vb_forward_protein, vb_md_eval, vb_md_run) ends with the all-reduce as ONE more kernel of its
 * CUDA graph: peer stores into every rank's window, a system-scope flag per sender, a fixed-order sum (bit-identical on
 * all ranks).  Option "comm_auto" 0 turns the automatic step off; vb_comm_allreduce runs it on any device buffer.
 * Replaces: the host-side gather of the per-device results (ThreadPoolExecutor + numpy concatenation,
 *           src/Calculators/bonded.py:74-89) ahead of combiner.py:38-39, and the NCCL all-reduce a caller would
 *           otherwise enqueue from the host every step.  Needs peer access between the GPUs (NVLink / NVSwitch). */
int vb_comm_init(vb_handle* h, int rank, int world, int64_t max_floats, void* ipc_handle_out /* 64 bytes */);
int vb_comm_connect(vb_handle* h, const void* all_handles /* world x 64 bytes, rank order */);
int vb_comm_allreduce(vb_handle* h, float* buf_dev, int64_t n, void* stream);

/* Copy the current neighbour list to the host: slots[N*32] (source index or -1), deg[N].
 * Replaces: the edge_index returned by torch_cluster.radius_graph at src/ViSNet/model/utils.py:260-266. */
int vb_get_edges(vb_handle* h, int32_t* slots_host, int32_t* deg_host);

/* Number of kernel launches of one vb_forward(), and whether it replays a captured CUDA graph. */
int vb_launches_per_forward(const vb_handle* h);
/* Tuning knobs: "use_graph" 0/1, "use_pdl" 0/1 (programmatic dependent launch between the stages, default off), "npw" 1/2, "te_fwd" 32/64, "te_bwd" 32/64, "node_impl" 0/1,
 * "edge_tc" bit0 = forward / bit1 = adjoint edge stage on tcgen05, "tc_rows" 32/64/96/128 fixed edges per tcgen05 tile
 * (0 = default: tile length planned so the tiles fill whole waves of CTAs, from an estimate of 17 edges per atom or,
 * after "calibrate" 1, from the edge count of the last evaluation -- synchronises), "timeline" 0/1 in-kernel phase stamps of the tcgen05 edge kernels and the SIMT node kernels (vb_debug_read "TL" / "TLN"),
 * "fused" 0/1 one launch per layer and direction (edge stage + node stage of a 4-node block; default off), "node_tc" 0/1
 * node stage on tcgen05 (default: from 600 atoms), "node_nb" 0/1/2/3/4/8 nodes per CTA of the SIMT node kernels (0 = the
 * fewest that fit one wave), "krot" 0/1 every CTA of the SIMT node kernels walks the K dimension of its weight chunks from a
 * different row (default 1: the CTAs of a wave otherwise ask the same L2 slices for the same rows at the same time),
 * "embed_batch" -1/0..3 batch variants of the embedding kernels, "comm_auto" 0/1.  vb_get_option also answers "edge_overflow" (1 after a step exceeded a trimmed max_edges),
 * "tile_rows" (planned edges per tile), "comm_ready", "caph_ready", "caph_evals" (energy evaluations of the last hydrogen refinement)
 * and "restraints_ready" (1 while a non-empty restraint set is installed). */
int vb_set_option(vb_handle* h, const char* key, int64_t value);
int64_t vb_get_option(const vb_handle* h, const char* key);   /* resolved value (after vb_set_topology) */

/* ---- diagnostics (stage-by-stage parity checks; not part of the hot path) ---- */
int vb_num_stages(const vb_handle* h);
const char* vb_stage_name(const vb_handle* h, int stage);
/* Run only the first n_stages launches of an evaluation, synchronously (no graph). */
int vb_debug_run(vb_handle* h, const float* pos_dev, int n_stages);
/* Per-launch device time (ms, CUDA events on the launching stream, average of n_iter eager evaluations after
 * one warm-up) for each of the vb_num_stages() launches; used by bench.py for the live roofline numbers. */
int vb_profile_stages(vb_handle* h, const float* pos_dev, int n_iter, float* ms_per_stage_host);
/* Self-test of the tcgen05/TMEM/TMA GEMM pipeline: d[128][128] = a[128][128] * W^T, W given as a tensor-core
 * weight image (ai2bmd_b200.weights.tc_image); repeated `reps` times inside one launch; *ms_out = kernel time. */
int vb_tc_selftest(int device, const float* a_host, const float* img_host, float* d_host, int reps, float* ms_out);
/* Copy an internal buffer to the host.  name: "X","V","F","VN","QKV","V123","VDOT","TU","O" (per layer),
 * "XA","VA","GX","GVEC","GF","GXA","GQKV","GVNMSG","GTU","GQKV2","GVNMSG2","GTU2","geom","rbf","eacc","grbf","esrc","edst","rowptr",
 * "eatom","energy","forces".  Returns the number of bytes copied (<= cap_bytes) or a negative status. */
int64_t vb_debug_read(vb_handle* h, const char* name, int layer, void* host_dst, int64_t cap_bytes);

#ifdef __cplusplus
}
#endif
#endif /* VISNET_B200_H */
