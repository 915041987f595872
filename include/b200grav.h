/*
 * b200grav.h -- C ABI of libb200grav.so, the B200 (sm_100a) gravitational
 * force engine that sits behind the reference's IForceComputer plugin API.
 *
 * Plain C: opaque handle, plain pointers and sizes, int status on every call
 * (0 = ok, otherwise a b200_status / cudaError_t+1000 / ncclResult_t+2000 --
 * see b200_error_string).  Nothing throws.  No torch, no TensorRT, no CPU
 * fallback: every compute entry point fails with B200_ERR_NO_DEVICE when no
 * sm_100 GPU is usable.
 *
 * "_host" entry points take HOST pointers in the reference's IForceComputer
 * layout (positions float[3N] AoS xyz, masses float[N], forces float[3N];
 * /root/reference include/core/interfaces.hpp:31-40) and do H2D, kernels, D2H.
 * "_dev" entry points take DEVICE pointers and a cudaStream_t (as void*; NULL is
 * the legacy default stream, as in a kernel launch) and only enqueue work,
 * in the reference's device layout (float4 x,y,z,m positions; 3 floats per
 * particle for velocities and forces; src/physics/lambda_cdm_impl.cu:65-68).
 *
 * Each entry point cites the reference interface it replaces.
 */
#ifndef B200GRAV_H
#define B200GRAV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200GRAV_ABI_VERSION 2

typedef struct b200_ctx b200_ctx;

enum b200_status {
    B200_OK = 0,
    B200_ERR_INVALID = 1,      /* bad argument (null pointer, eps <= 0, n > capacity ...) */
    B200_ERR_NO_DEVICE = 2,    /* no CUDA device / not an sm_100 part */
    B200_ERR_STATE = 3,        /* call out of order (walk before build ...) */
    B200_ERR_NOMEM = 4,
    B200_ERR_UNSUPPORTED = 5
    /* 1000 + cudaError_t, 2000 + ncclResult_t, 3000 + cufftResult */
};

const char* b200_error_string(int status);
int b200_abi_version(void);

/* ---- context -------------------------------------------------------------
 * Replaces the per-object device state of the reference's computers:
 * TreeForceComputer::initialize_gpu_resources / cleanup_gpu_resources
 * (src/forces/tree_force_computer.cpp:349-408), BarnesHutTree ctor/dtor
 * (src/forces/barnes_hut_tree.cu:343-381), LambdaCDMSimulationImpl ctor/dtor
 * (src/physics/lambda_cdm_impl.cu:80-145).  device = ForceComputeParameters::
 * cuda_device_id (include/forces/force_computer_factory.hpp:39).  Scratch
 * grows on demand; max_particles is a sizing hint (0 = grow lazily).
 *
 * Concurrency: ONE call in flight per context.  The "_dev" entry points accept any stream, but they share the
 * context's scratch (source tiles, partial sums, the equal-mass flag, tree tables, the target order), so a second
 * call must be ordered after the first -- same stream, or an event between the two; a tree walk goes on the stream
 * its build was given.  Independent work runs on independent contexts (one per GPU, or several per GPU). */
int b200_ctx_create(int device, size_t max_particles, b200_ctx** out);
int b200_ctx_destroy(b200_ctx* ctx);
int b200_ctx_device(const b200_ctx* ctx);
int b200_ctx_sm_count(const b200_ctx* ctx);
/* The context's own (non-blocking) cudaStream_t, for hosts that do not bring one. */
void* b200_ctx_stream(const b200_ctx* ctx);
/* Blocks until all work queued on stream (NULL = the context's own stream) is done. */
int b200_ctx_sync(b200_ctx* ctx, void* stream);

/* ---- direct sum (rows D1-D3) ---------------------------------------------
 * acc_i = sum_j m_j d / (|d|^2 + eps^2)^{3/2}, d = x_j - x_i, G = 1; output is
 * ACCELERATION (what TreeForceComputer writes), overwritten.
 * box > 0 selects the periodic minimum-image variant of compute_forces_direct
 * (src/physics/lambda_cdm_kernels.cu:14-56); box == 0 is the open-boundary sum
 * of the CPU leaf loop (src/forces/tree_force_computer.cpp:312-347).
 *
 * _host replaces IForceComputer::compute_forces for "DirectForceComputer"
 * (include/core/interfaces.hpp:33-35; name reserved at
 * src/forces/force_computer_factory.cpp:40-43).  mass == NULL means unit mass. */
int b200_direct_forces_host(b200_ctx* ctx, const float* pos3, const float* mass,
                            float* acc3, size_t n, float eps, float box);
/* _dev replaces launch_force_computation (src/physics/lambda_cdm_kernels.cu:
 * 444-468) and launch_nbody_force_kernel (src/tensorrt/nbody_plugins.cu:175-191).
 * posm4: float4[n_sources]; targets are posm4[i0 .. i0+n_targets); acc3:
 * float[3*n_targets].  This is the target-sharded form used on >1 GPU. */
int b200_direct_forces_dev(b200_ctx* ctx, const void* posm4, size_t n_sources,
                           size_t i0, size_t n_targets, float eps, float box,
                           void* acc3, void* stream);
/* Tile-SoA source format of the direct-sum kernel: [tile][x|y|z|m][512] floats,
 * 8 KB per 512 sources (slots past n hold zero-mass sources).  One TMA bulk copy
 * per tile.  b200_tiles_bytes(n) bytes hold n particles. */
size_t b200_tiles_bytes(size_t n);
int b200_pack_tiles_dev(b200_ctx* ctx, const void* posm4, size_t n, void* tiles, void* stream);
/* Direct sum with the sources supplied as `n_parts` (<= 16) tile-SoA buffers of
 * part_len[p] particles each, concatenated in order.  Buffers may live on PEER
 * GPUs (NVLink-mapped, see b200_ipc_*): the kernel pulls its source tiles
 * straight over NVLink, so no all-gather precedes it.  Targets are local:
 * targets4 float4[n_targets], acc3 float[3*n_targets].  all_masses_equal != 0 is
 * the caller's promise that every source in every part has the same mass (the
 * ranks agree on it once, masses do not change during a run): the 11-op
 * equal-mass instance runs.  0 = general masses. */
int b200_direct_forces_parts_dev(b200_ctx* ctx, const void* const* parts,
                                 const size_t* part_len, int n_parts,
                                 const void* targets4, size_t n_targets,
                                 float eps, float box, int all_masses_equal,
                                 void* acc3, void* stream);

/* ---- energy diagnostic (SURVEY 8f N4) -----------------------------------------
 * Replaces compute_energy + launch_energy_computation
 * (src/physics/lambda_cdm_kernels.cu:338-408, 492-516) and
 * LambdaCDMSimulationImpl::compute_energy (src/physics/lambda_cdm_impl.cu:222-241).
 * The O(N^2) pair sum runs in the direct-sum kernel (potential instance: 7-8 lane-ops
 * + 1 MUFU per pair, FP64 outer sums) instead of one thread per particle looping over
 * j > i from global memory.
 * phi_i = sum_{j != i} m_j / sqrt(|d|^2 + eps^2) >= 0 for targets posm4[i0..i0+n_targets);
 * box > 0: minimum image.  phi: float[n_targets] (device).  The pair loop has no self test;
 * the i == i term m_i/eps is subtracted afterwards, which leaves an absolute error of about
 * 1e-7 m_i/eps in phi_i (negligible unless phi_i << 1/eps, i.e. a handful of particles). */
int b200_direct_potential_dev(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0,
                              size_t n_targets, float eps, float box, void* phi, void* stream);
/* kinetic = sum 1/2 m v^2, potential = -1/2 sum m_i phi_i (G = 1) over the targets
 * [i0, i0+n_targets); vel3 = float[3*n_targets] (device, the targets' velocities).
 * Over all particles (i0 = 0, n_targets = n_sources) potential is the reference's
 * sum_{i<j} -m_i m_j / r.  On a sharded run each rank gets its share: add them
 * (b200_allreduce_sum_f64).  Blocks until the two HOST doubles are written. */
int b200_energy_dev(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0, size_t n_targets,
                    const void* vel3, float eps, float box, double* kinetic, double* potential,
                    void* stream);

/* Tree-vs-direct error measure of the reference's Barnes-Hut example
 * (examples/barnes_hut_test.cu:173-189): per particle |a_test - a_ref| / (|a_ref| + 1e-10),
 * its mean and its maximum over n particles; acc_*: float[3n] (device).  Blocking. */
int b200_force_error_dev(b200_ctx* ctx, const void* acc_test, const void* acc_ref, size_t n,
                         double* avg_rel_error, double* max_rel_error, void* stream);
/* Matter power spectrum of the particles, PowerSpectrumAnalyzer::compute_power_spectrum
 * (src/analysis/power_spectrum.cu:53-84) on the device: cloud-in-cell assignment on a grid^3
 * mesh (:86-134; positions taken modulo the box), density contrast (:161-180), forward FFT / grid^3
 * (cuFFT, bound at run time), shells of width 2 pi / box with half-spectrum multiplicities, x box^3,
 * optional subtraction of box^3 / grid^3 (:207-285).  Outputs (HOST, grid/2 entries each, any may be
 * NULL): bin centres k [h/Mpc], P(k) [(Mpc/h)^3], modes per bin.  Blocking. */
int b200_power_spectrum_dev(b200_ctx* ctx, const void* posm4, size_t n, int grid, float box,
                            int mass_weighted, int shot_noise_correction, float* k_out, float* p_out,
                            int* count_out, void* stream);

/* ---- periodic particle mesh ----------------------------------------------------
 * The solver the reference reserves the factory name "PMForceComputer" for (src/forces/
 * force_computer_factory.cpp:40-63) and never implements: the true periodic force of the box with a uniform
 * neutralising background, O(N + grid^3 log grid), where every other force path keeps only the nearest image.
 * Definition (G = 1; box L, mesh grid^3, h = L / grid, r_s = r_split):
 *   positions are wrapped, x - L floor(x / L) (the [0, L) and origin-centred frames give the same mesh); mesh point
 *   i sits at i h; cloud-in-cell (CIC) assignment of the sources posm4[0 .. n_sources) with masses .w;
 *   rho = sum m W / h^3 minus its mean (the k = 0 mode is zero);
 *   phi_k = -4 pi rho_k exp(-k^2 r_s^2) / (k^2 W(k)^2), W(k) = prod_a sinc^2(k_a h / 2)  (one W for the
 *   assignment, one for the interpolation, as GADGET-2);
 *   a_k = -i k_a phi_k (zero on the Nyquist plane of axis a), inverse FFT, CIC interpolation at the targets
 *   posm4[i0 .. i0+n_targets) with the deposit's weights.
 * acc3: float[3*n_targets] ACCELERATION, overwritten, in the sign convention of the direct sum.  phi (float
 * [n_targets], NULL = skip): the NEGATED mesh potential, interpolated the same way -- positive, as
 * b200_direct_potential_dev (potential energy = -1/2 sum m phi); long range only, and it includes the particle's
 * own smoothed self term (about m / (sqrt(pi) r_s)).
 * r_split > 0 is the Gaussian split radius of TreePM (Springel 2005); there is no "off" value, because without the
 * filter the W^-2 deconvolution makes the pair force noisy (100-200 % r.m.s. at 2-8 cells).  Recommended:
 * r_split = 1.25 h.  The PM force plus the short-range remainder sum m d / r^3 [erfc(r / 2 r_s) + r / (r_s sqrt(pi))
 * exp(-r^2 / 4 r_s^2)] (minimum image) then matches an Ewald sum to 0.02 / 0.2 / 0.8 / 1.0 / 0.6 / 0.3 % r.m.s. at
 * r = 0.5 / 1 / 2 / 4 / 8 / 12 h; used alone, the PM force is smooth below a few cells, the mesh's resolution.
 * The mass deposit accumulates in int64 fixed point: the meshes, and so the result for a target, are bitwise the
 * same whatever the storage order of the sources and whichever target range is asked for.  Sharded use: every rank
 * passes the full all-gathered array (b200_allgather_sources_dev) and its own target range (b200_shard_range); the
 * deposit is replicated, so the meshes are bitwise identical on every rank and the concatenated result is that of
 * one call.  FFTs are cuFFT, bound at run time: B200_ERR_UNSUPPORTED if libcufft is absent.  Meshes and plans are
 * kept on the context per grid (about 40 grid^3 bytes).
 * B200_ERR_INVALID: grid odd or outside 8..1024, box <= 0, r_split <= 0, i0 + n_targets > n_sources, acc3 NULL. */
int b200_pm_forces_dev(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0, size_t n_targets,
                       int grid, float box, float r_split, void* acc3, void* phi /* NULL = skip */, void* stream);
/* Host-array form for "PMForceComputer" (IForceComputer::compute_forces): pos3 float[3n], mass float[n] or NULL
 * (= 1), acc3 float[3n]; all n particles are sources and targets.  Blocking. */
int b200_pm_forces_host(b200_ctx* ctx, const float* pos3, const float* mass /* NULL = 1 */, float* acc3,
                        size_t n, int grid, float box, float r_split);
/* With b200_set_timing on: CUDA-event times (ms) of the phases of the last b200_pm_forces_dev on this context --
 * [0] deposit (mesh clear, mass bound, deposit), [1] convert, [2] R2C, [3] k-space, [4] the C2R transforms,
 * [5] interpolation, [6] the whole call.  Synchronises; B200_ERR_STATE without a timed call. */
int b200_pm_phase_ms(b200_ctx* ctx, float ms[7]);

/* ---- Barnes-Hut (rows T1-T6) ----------------------------------------------
 * Morton keys: replaces compute_morton_codes_kernel + morton3D
 * (src/forces/barnes_hut_tree.cu:33-55, include/forces/barnes_hut_tree.hpp:11-27);
 * IEEE divide, so device keys equal the host function bit for bit. */
int b200_morton_keys_dev(b200_ctx* ctx, const void* posm4, size_t n, float box,
                         void* keys_u32, void* stream);
/* Stable ascending (key, index) sort: replaces thrust::sequence + sort_by_key
 * (src/forces/barnes_hut_tree.cu:358,383-401).  keys_in is not modified. */
int b200_sort_pairs_dev(b200_ctx* ctx, const void* keys_in_u32, size_t n,
                        void* keys_out_u32, void* perm_out_i32, void* stream);
/* Octree build + centre of mass: replaces TreeForceComputer::build_tree_cpu
 * (src/forces/tree_force_computer.cpp:130-243) -- same tree, node for node:
 * root cube centred on the origin with edge `box`, first leaf_cap arrivals stay
 * in a node when it splits, strict > octant test, float centre recurrence. */
int b200_tree_build_dev(b200_ctx* ctx, const void* posm4, size_t n, float box,
                        int leaf_cap, int max_depth, void* stream);
/* Walk: replaces compute_tree_forces / compute_force_on_particle
 * (src/forces/tree_force_computer.cpp:245-347): accept iff size/|com-x| < theta,
 * eps = 0.01f monopole and unit-mass leaf pairs.  Targets posm4[i0..i0+n_targets)
 * of the array the tree was built from. acc3: float[3*n_targets]. */
int b200_tree_walk_dev(b200_ctx* ctx, size_t i0, size_t n_targets, float theta,
                       void* acc3, void* stream);
/* The two phases the reference class exposes separately (include/forces/tree_force_computer.hpp:78-80,
 * build_tree / compute_tree_forces) on host arrays; the particles stay on the device in between.
 * b200_tree_walk_host walks all n particles of the last b200_tree_build_host; the packed particles sit in a
 * buffer only b200_tree_build_host / b200_tree_forces_fixed_host write, so other host entry points may be
 * called in between. */
int b200_tree_build_host(b200_ctx* ctx, const float* pos3, const float* mass, size_t n, float box,
                         int leaf_cap, int max_depth);
int b200_tree_walk_host(b200_ctx* ctx, float* acc3, size_t n, float theta);
/* IForceComputer::compute_forces for "TreeForceComputer" on host arrays. */
int b200_tree_forces_host(b200_ctx* ctx, const float* pos3, const float* mass,
                          float* acc3, size_t n, float theta, int leaf_cap,
                          int max_depth, float box);

/* "Fixed physics" Barnes-Hut (SURVEY 8f N2) -- NOT the reference's tree.  The CPU
 * TreeForceComputer keeps the first leaf_cap particles of a node where they are when it splits
 * (src/forces/tree_force_computer.cpp:144-171; ~30 % of the mass never becomes a source), sums leaf
 * pairs with unit masses (:253, :340), centres its root cube on the origin whatever the data
 * (:132-133) and hard-codes eps = 0.01 (:281, :334): at theta = 0.5 its force is 0.3 (relative L2)
 * away from the direct sum.  This mode keeps the octant rule, the child geometry, the centre-of-mass
 * pass and the opening criterion, and removes those four: splitting nodes pass every particle on,
 * leaf pairs use the sources' masses, the root cube is fitted to the data (centre = bounding-box
 * midpoint, edge = largest extent * 1.00001), eps is a parameter.  Same kernels, same walk
 * (b200_tree_walk_dev / _stats / _export / _counters apply).  Checked against the FP64 direct
 * sum: 1.3e-3 relative L2 at theta = 0.5, 7e-5 at theta = 0.2 (uniform, leaf_cap 8).
 * The node table of this mode holds N/2 internal nodes (typical trees need N/25); a pathological input
 * that needs more (many tight knots of leaf_cap + 1 particles) fails loudly: the walk fills its output
 * with NaN, b200_tree_stats / _export / b200_tree_forces_fixed_host return B200_ERR_NOMEM. */
int b200_tree_build_fixed_dev(b200_ctx* ctx, const void* posm4, size_t n, int leaf_cap,
                              int max_depth, float eps, void* stream);
/* Fixed-physics walks only: box > 0 takes every separation (cell and particle) to its nearest periodic
 * image, d -= box * round(d / box) -- the minimum image of the reference's GPU kernels
 * (src/physics/lambda_cdm_kernels.cu:39-41, src/forces/barnes_hut_tree.cu:247-254); a cell that reaches across
 * the half-box distance from the target is always opened, so the result converges to the minimum-image direct
 * sum as theta -> 0; no Ewald sum.  0 = open
 * boundary (default).  The reference-faithful tree is never periodic (the CPU TreeForceComputer is not). */
int b200_tree_set_periodic(b200_ctx* ctx, float box);
/* Energy diagnostic from the fixed-physics tree (after b200_tree_build_fixed_dev): the walk accumulating
 * phi_i = sum m / sqrt(|d|^2 + eps^2) -- M / r for an accepted cell -- so that compute_energy
 * (src/physics/lambda_cdm_kernels.cu:338-408) costs O(N log N) in a tree run instead of O(N^2).
 * phi: float[n_targets] (device), positive, i == i excluded.  theta <= 1/sqrt(3) (a target must not
 * accept a cell that contains itself), else B200_ERR_UNSUPPORTED; B200_ERR_UNSUPPORTED for the
 * reference-faithful tree (unit-mass leaves, orphans).  _energy_: kinetic = sum 1/2 m v^2, potential =
 * -1/2 sum m_i phi_i over the target range, two HOST doubles, blocking. */
int b200_tree_potential_dev(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, void* phi, void* stream);
int b200_tree_energy_dev(b200_ctx* ctx, size_t i0, size_t n_targets, const void* vel3, float theta,
                         double* kinetic, double* potential, void* stream);
int b200_tree_forces_fixed_host(b200_ctx* ctx, const float* pos3, const float* mass /* NULL = 1 */,
                                float* acc3, size_t n, float theta, int leaf_cap, int max_depth,
                                float eps);

/* ---- octant-sharded build + forest walk (multi-GPU Barnes-Hut, row e) -------------------------------------
 * The reference builds one tree per process from all particles (build_tree_cpu, tree_force_computer.cpp:130-142).
 * The subtrees under the 8 children of the root are independent of each other once the root has routed its
 * arrivals -- the orphan rule is per node -- so the build shards by octant with no change to the tree:
 * part p of n_parts (<= 8) owns octants [8p/n_parts, 8(p+1)/n_parts) of the root; b200_tree_build_part_dev runs
 * the root level over all n particles and every deeper level over the particles of its own octants only; the
 * other octants stay empty leaves in this part's tree (b200_tree_stats / _export describe the part).
 *
 * arrival_i32 (device int32[n], or NULL): the reference's tree depends on the ORDER in which particles are
 * inserted (:136-140, index order).  arrival[k] = storage slot of the k-th particle to insert decouples that
 * order from where the particles are stored: a run that keeps its particles in a space-filling order (compact
 * shards, coherent gathers; b200_spatial_order_dev) passes the inverse of its storage permutation and gets the
 * reference's tree, node for node.  Particle ids in everything derived from the build (stored lists of
 * b200_tree_export, walk targets) are STORAGE SLOTS.  NULL = particles are stored in insertion order.
 * n_parts == 1 builds the whole tree (b200_tree_build_dev with an arrival order).
 *
 * b200_tree_forest_publish makes the part's walk tables visible to all walkers: over NCCL when the context has a
 * communicator of exactly n_parts ranks with rank == part (b200_shard_init; collective: table sizes and level-1 centres of mass by a 160-byte
 * all-gather + host read-back, then two all-gathers of equal-sized slices: the node records and the leaf sources as
 * 4-byte storage slots, from which every rank rebuilds the other parts' pair rows out of the positions it holds --
 * posm4 must be the same complete array on every rank), otherwise into this context's own
 * slot (one process building the parts in turn -- it must rebuild and publish EVERY part after particles move).
 * When every part is current the root's centre of mass is merged from the parts' level-1 nodes in the
 * reference's order and rounding.  After that b200_tree_walk_dev / b200_tree_walk_list_dev on this context walk
 * the forest (a part alone is not a tree; B200_ERR_STATE while a part is missing or stale).
 * b200_tree_walk_list_dev walks an explicit target list: targets = posm4[list[t]], acc3[3t..] in LIST order, a
 * warp = 32 consecutive list entries (the caller chooses the grouping).
 * Forces, counters and per-target interaction sets are those of the unsharded build + walk. */
int b200_tree_build_part_dev(b200_ctx* ctx, const void* posm4, const void* arrival_i32, size_t n, float box,
                             int leaf_cap, int max_depth, int part, int n_parts, void* stream);
int b200_tree_forest_publish(b200_ctx* ctx, void* stream);
int b200_tree_walk_list_dev(b200_ctx* ctx, const void* list_i32, size_t n_list, float theta, void* acc3,
                            void* stream);
/* Merged root record of the published forest (host): {com x, y, z, M, -, -, cell edge, -}.  Synchronises. */
int b200_tree_forest_root(b200_ctx* ctx, float out[8]);
/* dst4[perm[k]] = src4[k] for k < n (float4 rows, device): puts particles stored in another order -- e.g. the
 * rank-major all-gather of Hilbert-owned shards -- back at their original indices, the order the build needs. */
int b200_scatter_rows_dev(b200_ctx* ctx, const void* src4, const void* perm_i32, size_t n, void* dst4,
                          void* stream);
/* out4[k] = src4[list[k]] (float4 rows) and out3[k] = src3[list[k]] (3-float rows), device. */
int b200_gather_rows_dev(b200_ctx* ctx, const void* src4, const void* src3, const void* list_i32, size_t n,
                         void* out4, void* out3, void* stream);

/* Tree introspection (TreeForceComputer::get_node_count / get_leaf_count /
 * get_tree_depth, src/forces/tree_force_computer.cpp:410-464) and a canonical
 * breadth-first export for the bit-exact topology check.  Sizes first, then
 * export into caller-allocated HOST arrays (any pointer may be NULL to skip):
 *   level i32[n_nodes], center f32[3*n_nodes], size f32[n_nodes],
 *   first_child i32[n_nodes] (-1 = leaf), arrivals i64[n_nodes],
 *   part_off i64[n_nodes+1], part_idx i32[n_stored] (leaf members / orphans in
 *   arrival order), mass f32[n_nodes], com f32[3*n_nodes]. */
int b200_tree_stats(b200_ctx* ctx, size_t* n_nodes, size_t* n_leaves,
                    size_t* depth, size_t* n_stored);
int b200_tree_export(b200_ctx* ctx, int32_t* level, float* center, float* size,
                     int32_t* first_child, int64_t* arrivals, int64_t* part_off,
                     int32_t* part_idx, float* mass, float* com);
/* Walk counters of the last b200_tree_walk_dev with counting enabled:
 * [0] nodes visited, [1] monopole, [2] leaf pair interactions. */
int b200_tree_set_counting(b200_ctx* ctx, int enabled);
int b200_tree_counters(b200_ctx* ctx, uint64_t counters[3]);
/* Lane utilisation of the same counting walk (the measurement behind bench.py's `useful_lane_frac`):
 * [0..2] as b200_tree_counters; [3] pair-row source slots issued (64 per packed row a warp executes --
 * [2] / [3] is the fraction of them some target wanted); [4] node-visit lanes issued (32 per record a
 * warp loads), [5] of those, lanes that were awake (took part in the accept test). */
int b200_tree_walk_stats(b200_ctx* ctx, uint64_t stats[6]);
/* 1 if the last build ran out of node slots (fixed-physics mode only; the reference tree is bounded by
 * n / leaf_cap splits): the walk of such a tree fills its output with NaN.  Synchronises. */
int b200_tree_overflowed(b200_ctx* ctx, int* overflowed);

/* ---- leapfrog (rows L1-L3) -------------------------------------------------
 * Replaces leapfrog_update / launch_leapfrog_update
 * (src/physics/lambda_cdm_kernels.cu:290-335, 470-490) and the kick/drift
 * sequencing of LambdaCDMSimulationImpl::step (src/physics/lambda_cdm_impl.cu:
 * 167-213) with ONE pass over the particles:
 *     n_kicks times: v += (acc*m) * (1/m) * dt_kick * (1/a^2)      (:307-318)
 *     if dt_drift != 0: x += v*dt_drift; x = fmodf(x + box, box)   (:321-333)
 * n_kicks = 2 fuses the closing half-kick of step s with the opening half-kick
 * of step s+1 (same scale factor a in between) and the drift that follows.
 * box <= 0 disables the wrap.  a is the scale factor (double, as :296). */
int b200_leapfrog_dev(b200_ctx* ctx, void* posm4, void* vel3, const void* acc3,
                      size_t n, int n_kicks, float dt_kick, double a,
                      float dt_drift, float box, void* stream);
/* Host-array form (core::IIntegrator::step, include/core/interfaces.hpp:42-49):
 * pos3/vel3 float[3n] updated in place, acc3 float[3n], mass float[n] or NULL (= 1). */
int b200_leapfrog_host(b200_ctx* ctx, float* pos3, float* vel3, const float* acc3,
                       const float* mass, size_t n, int n_kicks, float dt_kick, double a,
                       float dt_drift, float box);
/* CosmologyModel::hubble_parameter_a (include/physics/cosmology_model.hpp:49-61)
 * and LambdaCDMSimulationImpl::update_scale_factor (lambda_cdm_impl.cu:261-269);
 * host scalars, double precision. */
double b200_hubble_a(double a, double omega_m, double omega_k, double omega_lambda, double h);
double b200_scale_factor_step(double a, double dt, double omega_m, double omega_k,
                              double omega_lambda, double h);

/* ---- initial conditions (SURVEY 8f N3) ------------------------------------------
 * Zel'dovich particles on the device.  Everything the reference's
 * InitialConditionsGenerator defines is kept -- BBKS-form P(k) = k^n_s T^2 normalised to
 * sigma_8 (src/physics/initial_conditions.cpp:83-171), Carroll-et-al. growth factor and
 * f = Omega_m(a)^0.55 (include/physics/cosmology_model.hpp:79-97), cell-centre grid, flat
 * index i*G*G + j*G + k, wrap into [0, box), v = a H f D psi, unit masses, stride subsample
 * (:279-298, 334-380, 412-418) -- except its displacement step (:304-332), which skips the
 * inverse Fourier transform; here psi(x) is the inverse FFT of i k delta_k / k^2 (cuFFT,
 * bound at run time; B200_ERR_UNSUPPORTED if libcufft is absent).  White noise comes from
 * a counter-based hash of (seed, cell), so the field does not depend on launch shape. */
typedef struct b200_ic_params {
    int grid;                 /* G: grid points per dimension (even, 4..2048) */
    float box;                /* box edge, Mpc/h */
    double z_initial;
    uint32_t seed;
    double omega_m, omega_lambda, omega_k, h, sigma_8, n_s;
    float particle_mass;      /* written to posm4.w (<= 0 means 1) */
    float origin_shift;       /* subtracted from every coordinate after the wrap: box/2 gives the
                                 origin-centred convention of the CPU tree's root cube */
    int use_2lpt;             /* InitialConditionsParams::use_2lpt (initial_conditions.hpp:38): add the second-order
                                 displacement, x = q + D1 psi1 + D2 psi2 with lap phi2 = sum_{a<b}(phi1,aa phi1,bb -
                                 phi1,ab^2), psi2 = grad phi2, D2 = -3/7 D1^2 Omega_m^-1/143, v = a H (f1 D1 psi1 +
                                 f2 D2 psi2), f2 = 2 Omega_m^6/11 -- computed in real space with 10 more FFTs, not by
                                 the reference's 26-neighbour mode sum (initial_conditions.cpp:639-722) */
} b200_ic_params;
void b200_ic_params_default(b200_ic_params* p);   /* the reference's defaults: 256, 100, z 49, seed 12345, ... */
/* n_particles <= G^3: particle p is grid point p * max(1, G^3 / n_particles).
 * posm4: float4[n_particles], vel3: float[3*n_particles] (device).  stats (host, may be NULL):
 * [0] r.m.s. displacement, [1] largest displacement (Mpc/h), [2] growth factor D(a_init),
 * [3] a H f.  Blocking. */
int b200_zeldovich_ics_dev(b200_ctx* ctx, const b200_ic_params* params, size_t n_particles,
                           void* posm4, void* vel3, double stats[4], void* stream);

/* Space-filling-curve order of the particles (the role of morton_encode_3d in the reference's domain
 * decomposition, src/mpi/domain_decomposition.cpp:114-208): perm[k] = index of the k-th particle along a
 * Hilbert curve over the cube [-box/2, box/2)^3 (stable for equal keys).  A run that STORES its particles
 * in this order gives every rank of the target-sharded scheme a compact region of space -- the 2^24-particle
 * Barnes-Hut step on 8 GPUs drops from 15.6 to 9.8 ms -- and makes the build's gathers coalesce.
 * perm: int32[n] (device). */
int b200_spatial_order_dev(b200_ctx* ctx, const void* posm4, size_t n, float box, void* perm_i32, void* stream);

/* ---- layout helpers --------------------------------------------------------
 * pos3 + mass (device) -> float4 x,y,z,m (device); mass == NULL -> 1. */
int b200_pack_posm_dev(b200_ctx* ctx, const void* pos3, const void* mass, size_t n,
                       void* posm4, void* stream);

/* ---- multi-GPU (row e) -----------------------------------------------------
 * Target-sharded data parallelism: rank r owns targets [r*N/G, (r+1)*N/G);
 * sources are all-gathered (semantic ancestor: ClusterCommunicator::
 * gather_all_particles, src/mpi/cluster_comm.cpp:218-247) -- either by the
 * caller's NCCL (torch.distributed) or pulled over NVLink by
 * b200_direct_forces_parts_dev from peer buffers mapped with these calls.
 * handle is a 64-byte cudaIpcMemHandle_t. */
/* Shard bounds of rank `rank` of `world`: i0 = rank*n/world, n_local = (rank+1)*n/world - i0. */
int b200_shard_range(size_t n, int rank, int world, size_t* i0, size_t* n_local);
/* A communicator owned by the context, for hosts without one of their own (the C++
 * plugin side).  Rank 0 calls b200_shard_unique_id and hands the 128 bytes
 * (an ncclUniqueId) to the other ranks by any means (file, socket, MPI, threads of
 * one process); every rank then calls b200_shard_init on its own context/device.
 * NCCL is bound at run time (libnccl.so.2); B200_ERR_UNSUPPORTED if it is absent.
 * world == 1 needs no id and makes the all-gather a no-op. */
#define B200_SHARD_ID_BYTES 128
int b200_shard_unique_id(unsigned char id[B200_SHARD_ID_BYTES]);
int b200_shard_init(b200_ctx* ctx, const unsigned char id[B200_SHARD_ID_BYTES], int rank, int world);
int b200_shard_finalize(b200_ctx* ctx);
int b200_shard_info(const b200_ctx* ctx, int* rank, int* world);
/* In-place all-gather of the float4 (x,y,z,m) shards: posm4_full is float4[n_total] on
 * this rank's device with this rank's particles already at their b200_shard_range
 * slice; when the stream reaches this point every slice holds its owner's data.
 * Replaces ClusterCommunicator::gather_all_particles (src/mpi/cluster_comm.cpp:218-247:
 * MPI_Allgather of counts + MPI_Allgatherv of host structs) -- device buffers, NVLink,
 * no host staging.  Equal shards use one ncclAllGather; ragged ones a grouped
 * broadcast per owner. */
int b200_allgather_sources_dev(b200_ctx* ctx, void* posm4_full, size_t n_total, void* stream);
/* Sum `count` HOST doubles over the ranks of b200_shard_init (in place; blocking).
 * The scalar diagnostics' MPI_Allreduce (src/mpi/cluster_comm.cpp:208-216 reduces forces;
 * here only energies need it).  A no-op on an unsharded context. */
int b200_allreduce_sum_f64(b200_ctx* ctx, double* values, size_t count);

/* Page-locks a HOST range the caller owns for the lifetime of the registration (cudaHostRegister), so that the
 * _host entry points' copies run at DMA speed instead of through the driver's pageable staging (2^20-particle
 * tree evaluation: 4.2 ms -> 3.1 ms end to end).  For long-lived arrays only -- the engine's particle arrays
 * (simulation_engine.hpp:60-63) -- and never for memory that is freed while registered. */
int b200_host_register(b200_ctx* ctx, void* host_ptr, size_t bytes);
int b200_host_unregister(b200_ctx* ctx, void* host_ptr);

int b200_device_alloc(b200_ctx* ctx, size_t bytes, void** dev_ptr);   /* cudaMalloc: exportable */
int b200_device_free(b200_ctx* ctx, void* dev_ptr);
/* Stream-ordered copies for hosts that keep the state device-resident (the
 * cudaMemcpy calls of LambdaCDMSimulation::copy_*_to_host, lambda_cdm_impl.cu).
 * d2h blocks until the data has arrived; h2d is asynchronous for pinned memory. */
int b200_memcpy_h2d(b200_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes, void* stream);
int b200_memcpy_d2h(b200_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes, void* stream);
/* posm4 (device) -> pos3 (device), the inverse of b200_pack_posm_dev */
int b200_unpack_pos3_dev(b200_ctx* ctx, const void* posm4, size_t n, void* pos3, void* stream);
int b200_ipc_export(b200_ctx* ctx, void* dev_ptr, unsigned char handle[64]);
int b200_ipc_open(b200_ctx* ctx, const unsigned char handle[64], void** dev_ptr);
int b200_ipc_close(b200_ctx* ctx, void* dev_ptr);

/* ---- measurement -----------------------------------------------------------
 * FP32 pipe probe for the roofline denominator (MEASURED_PEAKS.json has no
 * FP32 number): runs a register-resident FFMA chain on every SM and returns
 * achieved TFLOP/s (2 flop per FMA lane).  mode 0 = FFMA, 1 = FFMA2 (f32x2). */
int b200_fp32_peak_probe(b200_ctx* ctx, int mode, int iters, double* tflops, float* ms);
/* Device time (ms) of the last direct / tree call's main kernel, measured with
 * CUDA events on the stream it ran on; and the number of kernel launches this
 * context has issued since creation. */
int b200_last_kernel_ms(b200_ctx* ctx, float* ms);
int b200_set_timing(b200_ctx* ctx, int enabled);
uint64_t b200_launch_count(const b200_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
