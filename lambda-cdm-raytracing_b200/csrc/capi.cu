// capi.cu -- the extern "C" surface of libb200grav.so (include/b200grav.h).
#include <math.h>
#include <new>
#include <string.h>

#include "common.cuh"
#include "diag.cuh"
#include "direct.cuh"
#include "ics.cuh"
#include "leapfrog.cuh"
#include "pm.cuh"
#include "probe.cuh"
#include "shard.cuh"
#include "sort.cuh"
#include "tree.cuh"

using namespace b200;

// _dev entry points: `stream` is a cudaStream_t; NULL is CUDA's legacy default stream,
// exactly as in a kernel launch (so work ordered on the caller's default stream stays ordered).
static inline cudaStream_t pick_stream(b200_ctx*, void* stream) { return (cudaStream_t)stream; }

extern "C" {

const char* b200_error_string(int status) {
    switch (status) {
        case B200_OK: return "ok";
        case B200_ERR_INVALID: return "invalid argument";
        case B200_ERR_NO_DEVICE: return "no usable sm_100 CUDA device (there is no CPU fallback)";
        case B200_ERR_STATE: return "call out of order";
        case B200_ERR_NOMEM: return "device allocation failed";
        case B200_ERR_UNSUPPORTED: return "unsupported configuration";
        default: break;
    }
    if (status >= 1000 && status < 2000) return cudaGetErrorString((cudaError_t)(status - 1000));
    if (status >= 2000 && status < 3000) return shard_error_string(status - 2000);
    if (status >= 3000 && status < 4000) return "cuFFT error (status - 3000 is the cufftResult)";
    return "unknown b200grav status";
}

int b200_abi_version(void) { return B200GRAV_ABI_VERSION; }

int b200_ctx_create(int device, size_t max_particles, b200_ctx** out) {
    if (!out) return B200_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return B200_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) return B200_ERR_INVALID;
    cudaDeviceProp prop;
    B200_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return B200_ERR_NO_DEVICE;     // sm_100a SASS only
    B200_CUDA(cudaSetDevice(device));
    b200_ctx* ctx = new (std::nothrow) b200_ctx();
    if (!ctx) return B200_ERR_NOMEM;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    cudaError_t ce = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaEventCreate(&ctx->ev0);
    if (ce == cudaSuccess) ce = cudaEventCreate(&ctx->ev1);
    if (ce != cudaSuccess) { b200_ctx_destroy(ctx); return 1000 + (int)ce; }
    if (max_particles) {
        int s = ctx->src_tiles.reserve(direct_tiles_bytes(max_particles));
        if (s != B200_OK) { b200_ctx_destroy(ctx); return s; }
    }
    *out = ctx;
    return B200_OK;
}

int b200_ctx_destroy(b200_ctx* ctx) {
    if (!ctx) return B200_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    tree_destroy(ctx);
    shard_finalize(ctx);
    pm_destroy(ctx);
    ctx->src_tiles.release(); ctx->partials.release(); ctx->mass_flag.release(); ctx->zero_flag.release();
    ctx->energy_part.release(); ctx->energy_phi.release(); ctx->energy_out.release();
    ctx->ic_wk.release(); ctx->ic_tmp.release(); ctx->ic_psi.release(); ctx->ic_stats.release();
    ctx->h_pos3.release(); ctx->h_vel3.release(); ctx->h_mass.release(); ctx->h_posm4.release(); ctx->h_acc3.release();
    ctx->h_tree_posm4.release();
    ctx->probe.release(); ctx->sort_scratch.release();
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return B200_OK;
}

int b200_ctx_device(const b200_ctx* ctx) { return ctx ? ctx->device : -1; }
int b200_ctx_sm_count(const b200_ctx* ctx) { return ctx ? ctx->sm_count : 0; }

void* b200_ctx_stream(const b200_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int b200_ctx_sync(b200_ctx* ctx, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaStreamSynchronize(stream ? (cudaStream_t)stream : ctx->stream));
    return B200_OK;
}

// ---- direct ---------------------------------------------------------------
int b200_direct_forces_dev(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0,
                           size_t n_targets, float eps, float box, void* acc3, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    if (n_targets == 0) return B200_OK;
    if (!posm4 || !acc3 || i0 + n_targets > n_sources) return B200_ERR_INVALID;
    if (!(eps > 0.f) || box < 0.f) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = pick_stream(ctx, stream);
    B200_TRY(ctx->src_tiles.reserve(direct_tiles_bytes(n_sources)));
    B200_TRY(ctx->mass_flag.reserve(sizeof(int)));
    B200_TRY(direct_pack_tiles(ctx, posm4, n_sources, ctx->src_tiles.as<float>(), ctx->mass_flag.as<int>(), st));
    DirectSources src;
    memset(&src, 0, sizeof src);
    src.n_parts = 1;
    src.tiles[0] = ctx->src_tiles.as<float>();
    src.total_tiles = src.tile_end[0] = (int)((n_sources + DIRECT_TILE_J - 1) / DIRECT_TILE_J);
    return direct_forces(ctx, src, (const float4*)posm4 + i0, n_targets, eps, box, acc3,
                         ctx->mass_flag.as<int>(), st);
}

// ---- energy diagnostic ---------------------------------------------------------
int b200_direct_potential_dev(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0,
                              size_t n_targets, float eps, float box, void* phi, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    if (n_targets == 0) return B200_OK;
    if (!posm4 || !phi || i0 + n_targets > n_sources) return B200_ERR_INVALID;
    if (!(eps > 0.f) || box < 0.f) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = pick_stream(ctx, stream);
    B200_TRY(ctx->src_tiles.reserve(direct_tiles_bytes(n_sources)));
    B200_TRY(ctx->mass_flag.reserve(sizeof(int)));
    B200_TRY(direct_pack_tiles(ctx, posm4, n_sources, ctx->src_tiles.as<float>(), ctx->mass_flag.as<int>(), st));
    DirectSources src;
    memset(&src, 0, sizeof src);
    src.n_parts = 1;
    src.tiles[0] = ctx->src_tiles.as<float>();
    src.total_tiles = src.tile_end[0] = (int)((n_sources + DIRECT_TILE_J - 1) / DIRECT_TILE_J);
    return direct_potential(ctx, src, (const float4*)posm4 + i0, n_targets, eps, box, phi,
                            ctx->mass_flag.as<int>(), st);
}

int b200_energy_dev(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0, size_t n_targets,
                    const void* vel3, float eps, float box, double* kinetic, double* potential,
                    void* stream) {
    if (!ctx || !kinetic || !potential) return B200_ERR_INVALID;
    *kinetic = *potential = 0.0;
    if (n_targets == 0) return B200_OK;
    if (!posm4 || !vel3 || i0 + n_targets > n_sources) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = pick_stream(ctx, stream);
    B200_TRY(ctx->energy_phi.reserve(n_targets * sizeof(float)));
    B200_TRY(ctx->energy_out.reserve(2 * sizeof(double)));
    B200_TRY(b200_direct_potential_dev(ctx, posm4, n_sources, i0, n_targets, eps, box, ctx->energy_phi.p, stream));
    B200_TRY(energy_reduce(ctx, (const float4*)posm4 + i0, vel3, ctx->energy_phi.p, n_targets,
                           ctx->energy_out.as<double>(), st));
    double h[2];
    B200_CUDA(cudaMemcpyAsync(h, ctx->energy_out.p, sizeof h, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    *kinetic = h[0];
    *potential = h[1];
    return B200_OK;
}

int b200_force_error_dev(b200_ctx* ctx, const void* acc_test, const void* acc_ref, size_t n,
                         double* avg_rel_error, double* max_rel_error, void* stream) {
    if (!ctx || !avg_rel_error || !max_rel_error) return B200_ERR_INVALID;
    *avg_rel_error = *max_rel_error = 0.0;
    if (n == 0) return B200_OK;
    if (!acc_test || !acc_ref) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return force_error(ctx, acc_test, acc_ref, n, avg_rel_error, max_rel_error, pick_stream(ctx, stream));
}

int b200_power_spectrum_dev(b200_ctx* ctx, const void* posm4, size_t n, int grid, float box,
                            int mass_weighted, int shot_noise_correction, float* k_out, float* p_out,
                            int* count_out, void* stream) {
    if (!ctx || !posm4 || n == 0 || grid < 4 || (grid & 1) || grid > 2048 || !(box > 0.f)) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    const int s = power_spectrum(ctx, posm4, n, grid, box, mass_weighted, shot_noise_correction, k_out, p_out,
                                 count_out, pick_stream(ctx, stream));
    ctx->ic_wk.release(); ctx->ic_psi.release();        // two G^3 arrays: a one-off
    return s;
}

size_t b200_tiles_bytes(size_t n) { return direct_tiles_bytes(n); }

int b200_pack_tiles_dev(b200_ctx* ctx, const void* posm4, size_t n, void* tiles, void* stream) {
    if (!ctx || (n && (!posm4 || !tiles))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return direct_pack_tiles(ctx, posm4, n, (float*)tiles, nullptr, pick_stream(ctx, stream));
}

int b200_direct_forces_parts_dev(b200_ctx* ctx, const void* const* parts, const size_t* part_len,
                                 int n_parts, const void* targets4, size_t n_targets, float eps,
                                 float box, int all_masses_equal, void* acc3, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    if (n_targets == 0) return B200_OK;
    if (!parts || !part_len || n_parts < 1 || n_parts > DIRECT_MAX_PARTS || !targets4 || !acc3)
        return B200_ERR_INVALID;
    if (!(eps > 0.f) || box < 0.f) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    DirectSources src;
    memset(&src, 0, sizeof src);
    int total = 0, np = 0;
    for (int p = 0; p < n_parts; ++p) {
        int nt = (int)((part_len[p] + DIRECT_TILE_J - 1) / DIRECT_TILE_J);
        if (nt == 0) continue;
        if (!parts[p]) return B200_ERR_INVALID;
        total += nt;
        src.tiles[np] = (const float*)parts[p];
        src.tile_end[np] = total;
        ++np;
    }
    src.n_parts = np;
    src.total_tiles = total;
    const int* flag = nullptr;
    if (all_masses_equal) {         // a device int that reads 0 = "no source differs from the first"
        B200_TRY(ctx->zero_flag.reserve(sizeof(int)));
        B200_CUDA(cudaMemsetAsync(ctx->zero_flag.p, 0, sizeof(int), pick_stream(ctx, stream)));
        flag = ctx->zero_flag.as<int>();
    }
    return direct_forces(ctx, src, targets4, n_targets, eps, box, acc3, flag, pick_stream(ctx, stream));
}

int b200_direct_forces_host(b200_ctx* ctx, const float* pos3, const float* mass, float* acc3,
                            size_t n, float eps, float box) {
    if (!ctx) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;            // tree_force_computer.cpp:83
    if (!pos3 || !acc3) return B200_ERR_INVALID;
    if (!(eps > 0.f) || box < 0.f) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    B200_TRY(ctx->h_pos3.reserve(n * 3 * sizeof(float)));
    B200_TRY(ctx->h_posm4.reserve(n * 4 * sizeof(float)));
    B200_TRY(ctx->h_acc3.reserve(n * 3 * sizeof(float)));
    B200_CUDA(cudaMemcpyAsync(ctx->h_pos3.p, pos3, n * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
    const float* d_mass = nullptr;
    if (mass) {
        B200_TRY(ctx->h_mass.reserve(n * sizeof(float)));
        B200_CUDA(cudaMemcpyAsync(ctx->h_mass.p, mass, n * sizeof(float), cudaMemcpyHostToDevice, st));
        d_mass = ctx->h_mass.as<float>();
    }
    B200_TRY(pack_posm(ctx, ctx->h_pos3.p, d_mass, n, ctx->h_posm4.p, st));
    B200_TRY(b200_direct_forces_dev(ctx, ctx->h_posm4.p, n, 0, n, eps, box, ctx->h_acc3.p, st));
    B200_CUDA(cudaMemcpyAsync(acc3, ctx->h_acc3.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

// ---- periodic particle mesh -------------------------------------------------
int b200_pm_forces_dev(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0, size_t n_targets,
                       int grid, float box, float r_split, void* acc3, void* phi, void* stream) {
    if (!ctx || !acc3 || i0 + n_targets > n_sources || (n_sources && !posm4)) return B200_ERR_INVALID;
    if (grid < 8 || grid > 1024 || (grid & 1) || !(box > 0.f) || !(r_split > 0.f)) return B200_ERR_INVALID;
    if (n_targets == 0) return B200_OK;
    B200_CUDA(cudaSetDevice(ctx->device));
    return pm_forces(ctx, posm4, n_sources, i0, n_targets, grid, box, r_split, acc3, phi, pick_stream(ctx, stream));
}

int b200_pm_forces_host(b200_ctx* ctx, const float* pos3, const float* mass, float* acc3, size_t n, int grid,
                        float box, float r_split) {
    if (!ctx || !acc3 || (n && !pos3)) return B200_ERR_INVALID;
    if (grid < 8 || grid > 1024 || (grid & 1) || !(box > 0.f) || !(r_split > 0.f)) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    B200_TRY(ctx->h_pos3.reserve(n * 3 * sizeof(float)));
    B200_TRY(ctx->h_posm4.reserve(n * 4 * sizeof(float)));
    B200_TRY(ctx->h_acc3.reserve(n * 3 * sizeof(float)));
    B200_CUDA(cudaMemcpyAsync(ctx->h_pos3.p, pos3, n * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
    const float* d_mass = nullptr;
    if (mass) {
        B200_TRY(ctx->h_mass.reserve(n * sizeof(float)));
        B200_CUDA(cudaMemcpyAsync(ctx->h_mass.p, mass, n * sizeof(float), cudaMemcpyHostToDevice, st));
        d_mass = ctx->h_mass.as<float>();
    }
    B200_TRY(pack_posm(ctx, ctx->h_pos3.p, d_mass, n, ctx->h_posm4.p, st));
    B200_TRY(pm_forces(ctx, ctx->h_posm4.p, n, 0, n, grid, box, r_split, ctx->h_acc3.p, nullptr, st));
    B200_CUDA(cudaMemcpyAsync(acc3, ctx->h_acc3.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_pm_phase_ms(b200_ctx* ctx, float ms[7]) {
    if (!ctx || !ms) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return pm_phase_ms(ctx, ms);
}

// ---- Barnes-Hut -------------------------------------------------------------
int b200_morton_keys_dev(b200_ctx* ctx, const void* posm4, size_t n, float box, void* keys_u32,
                         void* stream) {
    if (!ctx || (n && (!posm4 || !keys_u32))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return morton_keys(ctx, posm4, n, box, (uint32_t*)keys_u32, pick_stream(ctx, stream));
}

int b200_sort_pairs_dev(b200_ctx* ctx, const void* keys_in_u32, size_t n, void* keys_out_u32,
                        void* perm_out_i32, void* stream) {
    if (!ctx || (n && (!keys_in_u32 || !keys_out_u32 || !perm_out_i32))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    B200_TRY(ctx->sort_scratch.reserve(sort_scratch_bytes(n)));
    return sort_pairs(ctx, (const uint32_t*)keys_in_u32, n, (uint32_t*)keys_out_u32,
                      (int32_t*)perm_out_i32, 32, ctx->sort_scratch.p, pick_stream(ctx, stream));
}

int b200_spatial_order_dev(b200_ctx* ctx, const void* posm4, size_t n, float box, void* perm_i32, void* stream) {
    if (!ctx || (n && (!posm4 || !perm_i32)) || !(box > 0.f)) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = pick_stream(ctx, stream);
    B200_TRY(ctx->h_mass.reserve(2 * n * sizeof(uint32_t)));           // keys in / keys out
    B200_TRY(ctx->sort_scratch.reserve(sort_scratch_bytes(n)));
    uint32_t* keys = ctx->h_mass.as<uint32_t>();
    B200_TRY(hilbert_keys(ctx, posm4, n, box, nullptr, keys, st));
    return sort_pairs(ctx, keys, n, keys + n, (int32_t*)perm_i32, 30, ctx->sort_scratch.p, st);
}

int b200_tree_build_dev(b200_ctx* ctx, const void* posm4, size_t n, float box, int leaf_cap,
                        int max_depth, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_build(ctx, posm4, n, box, leaf_cap, max_depth, false, 0.01f, pick_stream(ctx, stream));
}

int b200_tree_build_fixed_dev(b200_ctx* ctx, const void* posm4, size_t n, int leaf_cap, int max_depth,
                              float eps, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_build(ctx, posm4, n, 0.f, leaf_cap, max_depth, true, eps, pick_stream(ctx, stream));
}

int b200_tree_forces_fixed_host(b200_ctx* ctx, const float* pos3, const float* mass, float* acc3, size_t n,
                                float theta, int leaf_cap, int max_depth, float eps) {
    if (!ctx) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    if (!pos3 || !acc3) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    B200_TRY(ctx->h_pos3.reserve(n * 3 * sizeof(float)));
    B200_TRY(ctx->h_posm4.reserve(n * 4 * sizeof(float)));
    B200_TRY(ctx->h_acc3.reserve(n * 3 * sizeof(float)));
    B200_CUDA(cudaMemcpyAsync(ctx->h_pos3.p, pos3, n * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
    const float* d_mass = nullptr;
    if (mass) {
        B200_TRY(ctx->h_mass.reserve(n * sizeof(float)));
        B200_CUDA(cudaMemcpyAsync(ctx->h_mass.p, mass, n * sizeof(float), cudaMemcpyHostToDevice, st));
        d_mass = ctx->h_mass.as<float>();
    }
    B200_TRY(ctx->h_tree_posm4.reserve(n * 4 * sizeof(float)));
    B200_TRY(pack_posm(ctx, ctx->h_pos3.p, d_mass, n, ctx->h_tree_posm4.p, st));
    B200_TRY(tree_build(ctx, ctx->h_tree_posm4.p, n, 0.f, leaf_cap, max_depth, true, eps, st));
    B200_TRY(tree_walk(ctx, 0, n, theta, ctx->h_acc3.p, st));
    B200_CUDA(cudaMemcpyAsync(acc3, ctx->h_acc3.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    int overflow = 0;
    B200_TRY(tree_overflowed(ctx, &overflow));
    return overflow ? B200_ERR_NOMEM : B200_OK;      // the walk has filled acc3 with NaN
}

int b200_tree_walk_dev(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, void* acc3,
                       void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_walk(ctx, i0, n_targets, theta, acc3, pick_stream(ctx, stream));
}

int b200_tree_build_part_dev(b200_ctx* ctx, const void* posm4, const void* arrival_i32, size_t n, float box,
                             int leaf_cap, int max_depth, int part, int n_parts, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_build_part(ctx, posm4, (const int*)arrival_i32, n, box, leaf_cap, max_depth, part, n_parts,
                           pick_stream(ctx, stream));
}

int b200_tree_forest_publish(b200_ctx* ctx, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_forest_publish(ctx, pick_stream(ctx, stream));
}

int b200_tree_walk_list_dev(b200_ctx* ctx, const void* list_i32, size_t n_list, float theta, void* acc3,
                            void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_walk_list(ctx, (const int*)list_i32, n_list, theta, acc3, pick_stream(ctx, stream));
}

int b200_tree_forest_root(b200_ctx* ctx, float out[8]) {
    if (!ctx || !out) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_forest_root(ctx, out);
}

int b200_scatter_rows_dev(b200_ctx* ctx, const void* src4, const void* perm_i32, size_t n, void* dst4, void* stream) {
    if (!ctx || (n && (!src4 || !perm_i32 || !dst4))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return scatter_rows(ctx, src4, perm_i32, n, dst4, pick_stream(ctx, stream));
}

int b200_gather_rows_dev(b200_ctx* ctx, const void* src4, const void* src3, const void* list_i32, size_t n,
                         void* out4, void* out3, void* stream) {
    if (!ctx || (n && !list_i32) || (src4 && !out4) || (src3 && !out3)) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return gather_rows(ctx, src4, src3, list_i32, n, out4, out3, pick_stream(ctx, stream));
}

int b200_host_register(b200_ctx* ctx, void* host_ptr, size_t bytes) {
    if (!ctx || !host_ptr || bytes == 0) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    const cudaError_t e = cudaHostRegister(host_ptr, bytes, cudaHostRegisterPortable);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return B200_OK; }
    B200_CUDA(e);
    return B200_OK;
}

int b200_host_unregister(b200_ctx* ctx, void* host_ptr) {
    if (!ctx || !host_ptr) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    const cudaError_t e = cudaHostUnregister(host_ptr);
    if (e == cudaErrorHostMemoryNotRegistered) { cudaGetLastError(); return B200_OK; }
    B200_CUDA(e);
    return B200_OK;
}

// The two phases of compute_forces as the reference class exposes them (tree_force_computer.hpp:78-80:
// build_tree / compute_tree_forces): the particles stay on the device between the calls.
int b200_tree_build_host(b200_ctx* ctx, const float* pos3, const float* mass, size_t n, float box,
                         int leaf_cap, int max_depth) {
    if (!ctx) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    if (!pos3 || !mass) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // The packed particles live in a buffer of their own (not the staging the other host entry points
    // reuse), so a direct / leapfrog host call between build_host and walk_host cannot clobber them.
    B200_TRY(ctx->h_pos3.reserve(n * 3 * sizeof(float)));
    B200_TRY(ctx->h_mass.reserve(n * sizeof(float)));
    B200_TRY(ctx->h_tree_posm4.reserve(n * 4 * sizeof(float)));
    B200_CUDA(cudaMemcpyAsync(ctx->h_pos3.p, pos3, n * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(ctx->h_mass.p, mass, n * sizeof(float), cudaMemcpyHostToDevice, st));
    B200_TRY(pack_posm(ctx, ctx->h_pos3.p, ctx->h_mass.p, n, ctx->h_tree_posm4.p, st));
    return tree_build(ctx, ctx->h_tree_posm4.p, n, box, leaf_cap, max_depth, false, 0.01f, st);
}

int b200_tree_walk_host(b200_ctx* ctx, float* acc3, size_t n, float theta) {
    if (!ctx) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    if (!acc3) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    B200_TRY(ctx->h_acc3.reserve(n * 3 * sizeof(float)));
    B200_TRY(tree_walk(ctx, 0, n, theta, ctx->h_acc3.p, st));
    B200_CUDA(cudaMemcpyAsync(acc3, ctx->h_acc3.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_tree_forces_host(b200_ctx* ctx, const float* pos3, const float* mass, float* acc3, size_t n,
                          float theta, int leaf_cap, int max_depth, float box) {
    if (!ctx) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;            // tree_force_computer.cpp:83
    if (!pos3 || !mass || !acc3) return B200_ERR_INVALID;
    B200_TRY(b200_tree_build_host(ctx, pos3, mass, n, box, leaf_cap, max_depth));
    return b200_tree_walk_host(ctx, acc3, n, theta);
}

int b200_tree_stats(b200_ctx* ctx, size_t* n_nodes, size_t* n_leaves, size_t* depth, size_t* n_stored) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_stats(ctx, n_nodes, n_leaves, depth, n_stored);
}

int b200_tree_export(b200_ctx* ctx, int32_t* level, float* center, float* size, int32_t* first_child,
                     int64_t* arrivals, int64_t* part_off, int32_t* part_idx, float* mass, float* com) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_export(ctx, level, center, size, first_child, arrivals, part_off, part_idx, mass, com);
}

int b200_tree_potential_dev(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, void* phi, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_potential(ctx, i0, n_targets, theta, phi, pick_stream(ctx, stream));
}

int b200_tree_energy_dev(b200_ctx* ctx, size_t i0, size_t n_targets, const void* vel3, float theta,
                         double* kinetic, double* potential, void* stream) {
    if (!ctx || !kinetic || !potential) return B200_ERR_INVALID;
    *kinetic = *potential = 0.0;
    if (n_targets == 0) return B200_OK;
    if (!vel3) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = pick_stream(ctx, stream);
    B200_TRY(ctx->energy_phi.reserve(n_targets * sizeof(float)));
    B200_TRY(ctx->energy_out.reserve(2 * sizeof(double)));
    B200_TRY(tree_potential(ctx, i0, n_targets, theta, ctx->energy_phi.p, st));
    B200_TRY(energy_reduce(ctx, (const float4*)tree_posm(ctx) + i0, vel3, ctx->energy_phi.p, n_targets,
                           ctx->energy_out.as<double>(), st));
    double h[2];
    B200_CUDA(cudaMemcpyAsync(h, ctx->energy_out.p, sizeof h, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    *kinetic = h[0];
    *potential = h[1];
    return B200_OK;
}

int b200_tree_set_periodic(b200_ctx* ctx, float box) {
    if (!ctx) return B200_ERR_INVALID;
    return tree_set_periodic(ctx, box);
}

int b200_tree_set_counting(b200_ctx* ctx, int enabled) {
    if (!ctx) return B200_ERR_INVALID;
    return tree_set_counting(ctx, enabled);
}

int b200_tree_counters(b200_ctx* ctx, uint64_t counters[3]) {
    if (!ctx || !counters) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_counters(ctx, counters);
}

int b200_tree_walk_stats(b200_ctx* ctx, uint64_t stats[6]) {
    if (!ctx || !stats) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_walk_stats(ctx, stats);
}

int b200_tree_overflowed(b200_ctx* ctx, int* overflowed) {
    if (!ctx || !overflowed) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return tree_overflowed(ctx, overflowed);
}

// ---- leapfrog ---------------------------------------------------------------
int b200_leapfrog_dev(b200_ctx* ctx, void* posm4, void* vel3, const void* acc3, size_t n,
                      int n_kicks, float dt_kick, double a, float dt_drift, float box, void* stream) {
    if (!ctx) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    if (!posm4 || !vel3 || !acc3) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return leapfrog(ctx, posm4, vel3, acc3, n, n_kicks, dt_kick, a, dt_drift, box,
                    pick_stream(ctx, stream));
}

int b200_leapfrog_host(b200_ctx* ctx, float* pos3, float* vel3, const float* acc3, const float* mass,
                       size_t n, int n_kicks, float dt_kick, double a, float dt_drift, float box) {
    if (!ctx) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    if (!pos3 || !vel3 || !acc3) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t b3 = n * 3 * sizeof(float);
    B200_TRY(ctx->h_pos3.reserve(b3));
    B200_TRY(ctx->h_posm4.reserve(n * 4 * sizeof(float)));
    B200_TRY(ctx->h_acc3.reserve(b3 + 16));
    B200_TRY(ctx->h_vel3.reserve(b3 + 16));
    B200_CUDA(cudaMemcpyAsync(ctx->h_pos3.p, pos3, b3, cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(ctx->h_vel3.p, vel3, b3, cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(ctx->h_acc3.p, acc3, b3, cudaMemcpyHostToDevice, st));
    const float* d_mass = nullptr;
    if (mass) {
        B200_TRY(ctx->h_mass.reserve(n * sizeof(float)));
        B200_CUDA(cudaMemcpyAsync(ctx->h_mass.p, mass, n * sizeof(float), cudaMemcpyHostToDevice, st));
        d_mass = ctx->h_mass.as<float>();
    }
    B200_TRY(pack_posm(ctx, ctx->h_pos3.p, d_mass, n, ctx->h_posm4.p, st));
    B200_TRY(leapfrog(ctx, ctx->h_posm4.p, ctx->h_vel3.p, ctx->h_acc3.p, n, n_kicks, dt_kick, a, dt_drift, box, st));
    B200_TRY(unpack_pos3(ctx, ctx->h_posm4.p, n, ctx->h_pos3.p, st));
    B200_CUDA(cudaMemcpyAsync(pos3, ctx->h_pos3.p, b3, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaMemcpyAsync(vel3, ctx->h_vel3.p, b3, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

// include/physics/cosmology_model.hpp:49-61: H(z) with a = 1/(1+z), z = 1/a - 1.
double b200_hubble_a(double a, double omega_m, double omega_k, double omega_lambda, double h) {
    const double z = 1.0 / a - 1.0;
    const double aa = 1.0 / (1.0 + z);
    const double e2 = omega_m * pow(aa, -3) + omega_k * pow(aa, -2) + omega_lambda;
    return 100.0 * h * sqrt(e2);
}

// src/physics/lambda_cdm_impl.cu:261-269: a += a * H(a) * dt (H in km/s/Mpc, as the reference).
double b200_scale_factor_step(double a, double dt, double omega_m, double omega_k,
                              double omega_lambda, double h) {
    return a + a * b200_hubble_a(a, omega_m, omega_k, omega_lambda, h) * dt;
}

int b200_pack_posm_dev(b200_ctx* ctx, const void* pos3, const void* mass, size_t n, void* posm4,
                       void* stream) {
    if (!ctx || (n && (!pos3 || !posm4))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return pack_posm(ctx, pos3, mass, n, posm4, pick_stream(ctx, stream));
}

// ---- initial conditions --------------------------------------------------------
void b200_ic_params_default(b200_ic_params* p) {
    if (!p) return;
    p->grid = 256;               // InitialConditionsParams defaults, initial_conditions.hpp:22-41
    p->box = 100.0f;
    p->z_initial = 49.0;
    p->seed = 12345u;
    p->omega_m = 0.31;           // CosmologyParams defaults, cosmology_model.hpp:11-18
    p->omega_lambda = 0.69;
    p->omega_k = 0.0;
    p->h = 0.67;
    p->sigma_8 = 0.81;
    p->n_s = 0.965;
    p->particle_mass = 1.0f;
    p->origin_shift = 0.0f;
    p->use_2lpt = 0;             // InitialConditionsParams::use_2lpt default (initial_conditions.hpp:38)
}

int b200_zeldovich_ics_dev(b200_ctx* ctx, const b200_ic_params* params, size_t n_particles, void* posm4,
                           void* vel3, double stats[4], void* stream) {
    if (!ctx || !params || !posm4 || !vel3) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    const int s = zeldovich_ics(ctx, params, n_particles, posm4, vel3, stats, pick_stream(ctx, stream));
    // three G^3 planes are a one-off: give them back
    ctx->ic_wk.release(); ctx->ic_tmp.release(); ctx->ic_psi.release();
    return s;
}

// ---- multi-GPU: NCCL source all-gather ---------------------------------------
int b200_shard_range(size_t n, int rank, int world, size_t* i0, size_t* n_local) {
    if (world < 1 || rank < 0 || rank >= world) return B200_ERR_INVALID;
    // 128-bit-safe form of [rank*n/world, (rank+1)*n/world)
    const size_t q = n / (size_t)world, r = n % (size_t)world;
    const size_t lo = (size_t)rank * q + ((size_t)rank * r) / (size_t)world;
    const size_t hi = (size_t)(rank + 1) * q + ((size_t)(rank + 1) * r) / (size_t)world;
    if (i0) *i0 = lo;
    if (n_local) *n_local = hi - lo;
    return B200_OK;
}

int b200_shard_unique_id(unsigned char id[B200_SHARD_ID_BYTES]) {
    if (!id) return B200_ERR_INVALID;
    return shard_unique_id(id);
}

int b200_shard_init(b200_ctx* ctx, const unsigned char id[B200_SHARD_ID_BYTES], int rank, int world) {
    if (!ctx || (world > 1 && !id)) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return shard_init(ctx, id, rank, world);
}

int b200_shard_finalize(b200_ctx* ctx) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    if (ctx->stream) B200_CUDA(cudaStreamSynchronize(ctx->stream));
    return shard_finalize(ctx);
}

int b200_shard_info(const b200_ctx* ctx, int* rank, int* world) {
    if (!ctx) return B200_ERR_INVALID;
    return shard_info(ctx, rank, world);
}

int b200_allreduce_sum_f64(b200_ctx* ctx, double* values, size_t count) {
    if (!ctx || (count && !values)) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return shard_allreduce_f64(ctx, values, count);
}

int b200_allgather_sources_dev(b200_ctx* ctx, void* posm4_full, size_t n_total, void* stream) {
    if (!ctx || (n_total && !posm4_full)) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return shard_allgather(ctx, posm4_full, n_total, pick_stream(ctx, stream));
}

// ---- multi-GPU peer mapping ------------------------------------------------
int b200_device_alloc(b200_ctx* ctx, size_t bytes, void** dev_ptr) {
    if (!ctx || !dev_ptr || bytes == 0) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    if (cudaMalloc(dev_ptr, bytes) != cudaSuccess) { cudaGetLastError(); return B200_ERR_NOMEM; }
    return B200_OK;
}

int b200_device_free(b200_ctx* ctx, void* dev_ptr) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    if (dev_ptr) B200_CUDA(cudaFree(dev_ptr));
    return B200_OK;
}

int b200_memcpy_h2d(b200_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes, void* stream) {
    if (!ctx || (bytes && (!dev_dst || !host_src))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    B200_CUDA(cudaMemcpyAsync(dev_dst, host_src, bytes, cudaMemcpyHostToDevice, pick_stream(ctx, stream)));
    return B200_OK;
}

int b200_memcpy_d2h(b200_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes, void* stream) {
    if (!ctx || (bytes && (!host_dst || !dev_src))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    B200_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, pick_stream(ctx, stream)));
    B200_CUDA(cudaStreamSynchronize(pick_stream(ctx, stream)));
    return B200_OK;
}

int b200_unpack_pos3_dev(b200_ctx* ctx, const void* posm4, size_t n, void* pos3, void* stream) {
    if (!ctx || (n && (!posm4 || !pos3))) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return unpack_pos3(ctx, posm4, n, pos3, pick_stream(ctx, stream));
}

int b200_ipc_export(b200_ctx* ctx, void* dev_ptr, unsigned char handle[64]) {
    if (!ctx || !dev_ptr || !handle) return B200_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    B200_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
    memcpy(handle, &h, 64);
    return B200_OK;
}

int b200_ipc_open(b200_ctx* ctx, const unsigned char handle[64], void** dev_ptr) {
    if (!ctx || !handle || !dev_ptr) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    B200_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return B200_OK;
}

int b200_ipc_close(b200_ctx* ctx, void* dev_ptr) {
    if (!ctx || !dev_ptr) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    B200_CUDA(cudaIpcCloseMemHandle(dev_ptr));
    return B200_OK;
}

// ---- measurement -------------------------------------------------------------
int b200_fp32_peak_probe(b200_ctx* ctx, int mode, int iters, double* tflops, float* ms) {
    if (!ctx) return B200_ERR_INVALID;
    B200_CUDA(cudaSetDevice(ctx->device));
    return fp32_peak_probe(ctx, mode, iters, tflops, ms);
}

int b200_set_timing(b200_ctx* ctx, int enabled) {
    if (!ctx) return B200_ERR_INVALID;
    ctx->timing = enabled != 0;
    return B200_OK;
}

int b200_last_kernel_ms(b200_ctx* ctx, float* ms) {
    if (!ctx || !ms) return B200_ERR_INVALID;
    if (!ctx->timing) return B200_ERR_STATE;
    B200_CUDA(cudaEventSynchronize(ctx->ev1));
    B200_CUDA(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return B200_OK;
}

uint64_t b200_launch_count(const b200_ctx* ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
