// sdp_b200.cu - hand-written sm_100a kernels + C ABI of the Bellman sweep engine.
//
// Hot path replaced (reference pierre-haessig/stodynprog, file:line relative to it):
//   * cell search + gather + nested lerp of multilinear_interpolation_{1..4}d
//     (stodynprog/dolointerpolation/multilinear_cython.pyx:54-300)
//   * the per-state backup _value_at_state_vect (stodynprog/stodynprog.py:639-691)
//     looped over the state grid by value_iteration (:511-515)
//   * the policy-evaluation iteration of eval_policy (:743-763)
// and adds the forward (transposed) application of a fixed policy's chain, which the
// reference has no counterpart for (K1'', distribution propagation).
//
// This is a gather-reduce, not a contraction: no tensor cores.  The sweep kernel
// streams the dense (cell, lambda, g) tables once from HBM with 128-bit
// streaming loads (ld.global.cs: evict-first, no reuse), gathers the 2^d corners
// of the previous value function through the read-only path (ld.global.nc, L1 +
// L2 resident: J is at most a few MB), accumulates the expectation over the
// perturbation nodes in registers in index order, and reduces (value, index)
// lexicographically over the control run with warp shuffles - one warp per work
// item (a state, or a run of controls of a state with many controls).
//
// Arithmetic contract (SURVEY.md App. A): fp64, round-to-nearest, explicit
// __dadd_rn/__dsub_rn/__dmul_rn/__ddiv_rn so that nvcc can never contract a
// multiply-add into an FMA; truncating cast with x86 cvttsd2si out-of-range
// semantics; weights are NOT clamped (linear extrapolation outside the grid).

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdarg.h>
#include <stdlib.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <limits.h>
#include <math.h>
#include <atomic>

#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>

#include "sdp_b200.h"

// ---------------------------------------------------------------------------
// error handling / accounting
// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

static int fail(int code, const char* fmt, const char* detail) {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}

#define SDP_CUDA_CHECK(expr)                                              \
    do {                                                                  \
        cudaError_t _e = (expr);                                          \
        if (_e != cudaSuccess)                                            \
            return fail(SDP_ECUDA, #expr ": %s", cudaGetErrorString(_e)); \
    } while (0)

#define SDP_LAUNCH_CHECK()                                                          \
    do {                                                                            \
        g_launches.fetch_add(1, std::memory_order_relaxed);                         \
        cudaError_t _e = cudaGetLastError();                                        \
        if (_e != cudaSuccess)                                                      \
            return fail(SDP_ECUDA, "kernel launch: %s", cudaGetErrorString(_e));    \
    } while (0)

extern "C" int sdp_version(void) { return SDP_ABI_VERSION; }
extern "C" const char* sdp_last_error(void) { return g_err; }
extern "C" int64_t sdp_launch_count(void) { return (int64_t)g_launches.load(); }

// name (template arguments, CTA shape) of the streaming kernel the calling thread's last
// sdp_sweep_partials launched: what a bench line or a profile summary should call it
static thread_local char g_last_kernel[192] = "";
static void note_kernel(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_kernel, sizeof(g_last_kernel), fmt, ap);
    va_end(ap);
}
extern "C" const char* sdp_last_kernel(void) { return g_last_kernel; }

// ---------------------------------------------------------------------------
// device-side grid description (kernel parameter, lives in constant bank)
// ---------------------------------------------------------------------------
template <typename T>
struct GridT {
    T smin[SDP_MAX_D];
    T span[SDP_MAX_D];    // smax - smin   (pyx: `(smax[k]-smin[k])`, recomputed per point there)
    T om1[SDP_MAX_D];     // (T)(order-1)
    int order[SDP_MAX_D];
    int stride[SDP_MAX_D];  // C-order strides M_k of the value array (pyx:109,164-165,235-237)
};

template <typename T>
static int make_grid(const SdpGrid* g, GridT<T>* out, int64_t* n_grid) {
    if (g == nullptr) return fail(SDP_EINVAL, "%s", "grid is NULL");
    if (g->d < 1 || g->d > SDP_MAX_D) return fail(SDP_EINVAL, "%s", "grid.d must be 1..4");
    int64_t n = 1;
    for (int k = g->d - 1; k >= 0; --k) {
        if (g->order[k] < 2)
            return fail(SDP_EINVAL, "%s", "every state axis needs at least 2 grid points");
        out->stride[k] = (int)n;
        n *= g->order[k];
        if (n >= (int64_t)INT_MAX) return fail(SDP_EINVAL, "%s", "grid has >= 2^31 points");
    }
    for (int k = 0; k < SDP_MAX_D; ++k) {
        if (k < g->d) {
            T lo = (T)g->smin[k], hi = (T)g->smax[k];
            out->smin[k] = lo;
            out->span[k] = hi - lo;
            out->om1[k] = (T)(g->order[k] - 1);
            out->order[k] = g->order[k];
        } else {
            out->smin[k] = 0; out->span[k] = 1; out->om1[k] = 1; out->order[k] = 2; out->stride[k] = 0;
        }
    }
    if (n_grid) *n_grid = n;
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// contraction-proof arithmetic
// ---------------------------------------------------------------------------
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double div_(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float add_(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float mul_(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float div_(float a, float b) { return __fdiv_rn(a, b); }

// C cast double->int as compiled for x86-64 (cvttsd2si): truncation toward zero;
// NaN and anything whose truncation does not fit int32 give INT_MIN ("integer
// indefinite"), which the reference then clamps to cell 0 (SURVEY.md App. A.2).
__device__ __forceinline__ int x86_trunc(double t) {
    if (!(t > -2147483649.0 && t < 2147483648.0)) return INT_MIN;
    return __double2int_rz(t);
}
__device__ __forceinline__ int x86_trunc(float t) {
    if (!(t >= -2147483648.0f && t < 2147483648.0f)) return INT_MIN;
    return __float2int_rz(t);
}

// cell index q and barycentric weight lam along one axis (pyx:117-131):
//   sn = (s - smin)/(smax - smin);  t = sn*(order-1)
//   q = max(min((int)t, order-2), 0);  lam = t - q
template <typename T>
__device__ __forceinline__ void cell_1d(T s, T smin, T span, T om1, int order, int& q, T& lam) {
    T sn = div_(sub_(s, smin), span);
    T t = mul_(sn, om1);
    int qi = x86_trunc(t);
    qi = max(min(qi, order - 2), 0);
    q = qi;
    lam = sub_(t, (T)qi);
}

// nested lerp, last axis innermost (pyx:88,140,208,300):
//   (1-l_K)*value(K+1 | corner 0) + l_K*value(K+1 | corner 1)
template <typename T, int D, int K>
struct Lerp {
    __device__ __forceinline__ static T eval(const T* __restrict__ V, int base,
                                             const int (&stride)[SDP_MAX_D], const T (&lam)[D]) {
        // the last axis has stride 1 (make_grid): a literal lets the two corner
        // loads share one address computation
        T a = Lerp<T, D, K + 1>::eval(V, base, stride, lam);
        T b = Lerp<T, D, K + 1>::eval(V, base + (K == D - 1 ? 1 : stride[K]), stride, lam);
        return add_(mul_(sub_((T)1, lam[K]), a), mul_(lam[K], b));
    }
};
template <typename T, int D>
struct Lerp<T, D, D> {
    __device__ __forceinline__ static T eval(const T* __restrict__ V, int base,
                                             const int (&)[SDP_MAX_D], const T (&)[D]) {
        return __ldg(V + base);
    }
};

// fp32 specialisation of the reference's fused type: the generated C writes the
// weights as `(1.0 - lam_k)` with a double literal, so the `(1.0-lam)*a` terms
// and the sums are evaluated in double while the innermost `lam*v` product of
// two floats stays a float product; one final rounding to float on the store.
template <int D, int K>
struct Lerp<float, D, K> {
    __device__ __forceinline__ static double eval_d(const float* __restrict__ V, int base,
                                                    const int (&stride)[SDP_MAX_D], const float (&lam)[D]) {
        if (K == D - 1) {
            float v0 = __ldg(V + base), v1 = __ldg(V + base + stride[K]);
            float t2 = mul_(lam[K], v1);
            return add_(mul_(sub_(1.0, (double)lam[K]), (double)v0), (double)t2);
        } else {
            double a = Lerp<float, D, (K + 1 < D ? K + 1 : K)>::eval_d(V, base, stride, lam);
            double b = Lerp<float, D, (K + 1 < D ? K + 1 : K)>::eval_d(V, base + stride[K], stride, lam);
            return add_(mul_(sub_(1.0, (double)lam[K]), a), mul_((double)lam[K], b));
        }
    }
    __device__ __forceinline__ static float eval(const float* __restrict__ V, int base,
                                                 const int (&stride)[SDP_MAX_D], const float (&lam)[D]) {
        return __double2float_rn(eval_d(V, base, stride, lam));
    }
};

// ---------------------------------------------------------------------------
// K0a: cell search on explicit points,  s [d][n] -> cell [n], lam [d][n]
// ---------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256)
k_cell_setup(GridT<double> G, int64_t n, const double* __restrict__ s,
             int32_t* __restrict__ cell, double* __restrict__ lam) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int base = 0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        int q; double l;
        cell_1d<double>(s[(int64_t)k * n + i], G.smin[k], G.span[k], G.om1[k], G.order[k], q, l);
        base += q * G.stride[k];
        lam[(int64_t)k * n + i] = l;
    }
    cell[i] = base;
}

extern "C" int sdp_cell_setup(const SdpGrid* grid, int64_t n, const double* s, int32_t* cell,
                              double* lam, void* stream) {
    GridT<double> G;
    int rc = make_grid<double>(grid, &G, nullptr);
    if (rc) return rc;
    if (n < 0 || (n > 0 && (!s || !cell || !lam))) return fail(SDP_EINVAL, "%s", "sdp_cell_setup: bad arguments");
    if (n == 0) return SDP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned blocks = (unsigned)((n + 255) / 256);
    switch (grid->d) {
        case 1: k_cell_setup<1><<<blocks, 256, 0, st>>>(G, n, s, cell, lam); break;
        case 2: k_cell_setup<2><<<blocks, 256, 0, st>>>(G, n, s, cell, lam); break;
        case 3: k_cell_setup<3><<<blocks, 256, 0, st>>>(G, n, s, cell, lam); break;
        default: k_cell_setup<4><<<blocks, 256, 0, st>>>(G, n, s, cell, lam); break;
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K0b: table build.  One thread per (state, w, u) entry; the fastest thread
// index follows the fastest table index so that the table writes are coalesced.
// ---------------------------------------------------------------------------
// source offset of element (flat control u, perturbation w) of slot k: the flat
// control index is decomposed C-order over the state's control grid dims
// (stodynprog.py:686 unravel_index), each axis with its own source stride.
__device__ __forceinline__ int64_t src_offset(const SdpStateDesc* ds, int k, int u, int w) {
    int64_t off = ds->src[k] + (int64_t)w * ds->ws[k];
#pragma unroll
    for (int c = SDP_MAX_C - 1; c >= 0; --c) {
        const int n = ds->npts[c];
        const int i = u % n;
        u /= n;
        off += (int64_t)i * ds->cs[k][c];
    }
    return off;
}

template <int D>
__device__ __forceinline__ void build_entry(const GridT<double>& G, const SdpStateDesc* ds, bool live,
                                            int u, int w, const double* __restrict__ staging,
                                            int32_t* __restrict__ cell, double* __restrict__ lam,
                                            int64_t lam_plane, int64_t off) {
    int base = 0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        double l = 0.0;
        if (live) {
            int q;
            double sk = staging[src_offset(ds, k, u, w)];
            cell_1d<double>(sk, G.smin[k], G.span[k], G.om1[k], G.order[k], q, l);
            base += q * G.stride[k];
        }
        lam[(int64_t)k * lam_plane + off] = l;
    }
    cell[off] = base;
}

template <int D>
__global__ void __launch_bounds__(256)
k_build_tables(GridT<double> G, int W, int g_per_w, int tiles_per_state,
               const SdpStateDesc* __restrict__ desc, const double* __restrict__ staging,
               int32_t* __restrict__ cell, double* __restrict__ lam, int64_t lam_plane,
               double* __restrict__ g) {
    const int64_t state = blockIdx.x / tiles_per_state;
    const int tile = blockIdx.x % tiles_per_state;
    const SdpStateDesc* ds = desc + state;
    const int Upad = ds->Upad;
    const int U = ds->U;
    const int e = tile * blockDim.x + threadIdx.x;  // entry within the block: w*Upad + u
    if (e >= W * Upad) return;
    const int w = e / Upad;
    const int u = e - w * Upad;
    const int64_t off = ds->entry_off + e;
    const bool live = u < U;
    build_entry<D>(G, ds, live, u, w, staging, cell, lam, lam_plane, off);
    if (g_per_w || w == 0) {
        double gv = 0.0;
        if (live) gv = staging[src_offset(ds, D, u, w)];
        g[ds->g_off + (g_per_w ? e : u)] = gv;
    }
}

extern "C" int sdp_build_tables(const SdpGrid* grid, int32_t W, int32_t g_per_w, int64_t n_states,
                                const SdpStateDesc* desc, const double* staging, int32_t* cell,
                                double* lam, int64_t lam_plane, double* g, int32_t max_Upad,
                                void* stream) {
    GridT<double> G;
    int rc = make_grid<double>(grid, &G, nullptr);
    if (rc) return rc;
    if (W < 1 || n_states < 0 || max_Upad < 0 || (max_Upad & 3))
        return fail(SDP_EINVAL, "%s", "sdp_build_tables: bad sizes");
    if (n_states == 0 || max_Upad == 0) return SDP_OK;
    if (!desc || !staging || !cell || !lam || !g) return fail(SDP_EINVAL, "%s", "sdp_build_tables: NULL pointer");
    int64_t per_state = (int64_t)W * max_Upad;
    int tiles = (int)((per_state + 255) / 256);
    int64_t blocks = n_states * tiles;
    if (blocks > 0x7fffffffLL) return fail(SDP_EINVAL, "%s", "sdp_build_tables: chunk too large");
    cudaStream_t st = (cudaStream_t)stream;
    switch (grid->d) {
        case 1: k_build_tables<1><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, tiles, desc, staging, cell, lam, lam_plane, g); break;
        case 2: k_build_tables<2><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, tiles, desc, staging, cell, lam, lam_plane, g); break;
        case 3: k_build_tables<3><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, tiles, desc, staging, cell, lam, lam_plane, g); break;
        default: k_build_tables<4><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, tiles, desc, staging, cell, lam, lam_plane, g); break;
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// layout B: entries of a tile are [u][w][lane]; thread e -> lane = e%32, (u,w) = e/32
template <int D>
__global__ void __launch_bounds__(256)
k_build_tables_tiled(GridT<double> G, int W, int g_per_w, int blocks_per_tile, int64_t n_states,
                     const SdpStateDesc* __restrict__ desc, const double* __restrict__ staging,
                     const int64_t* __restrict__ tile_off, const int64_t* __restrict__ tile_g_off,
                     const int32_t* __restrict__ tile_U, int32_t* __restrict__ cell,
                     double* __restrict__ lam, int64_t lam_plane, double* __restrict__ g) {
    const int64_t tile = blockIdx.x / blocks_per_tile;
    const int blk = blockIdx.x % blocks_per_tile;
    const int Ut = tile_U[tile];
    const int e = blk * blockDim.x + threadIdx.x;
    if (e >= Ut * W * 32) return;
    const int lane = e & 31;
    const int r = e >> 5;
    const int u = r / W;
    const int w = r - u * W;
    const int64_t state = tile * 32 + lane;
    const bool in_range = state < n_states;
    const SdpStateDesc* ds = desc + (in_range ? state : 0);
    const bool live = in_range && u < ds->U;
    const int64_t off = tile_off[tile] + e;
    build_entry<D>(G, ds, live, u, w, staging, cell, lam, lam_plane, off);
    if (g_per_w || w == 0) {
        double gv = 0.0;
        if (live) gv = staging[src_offset(ds, D, u, w)];
        g[g_per_w ? off : (tile_g_off[tile] + (int64_t)u * 32 + lane)] = gv;
    }
}

extern "C" int sdp_build_tables_tiled(const SdpGrid* grid, int32_t W, int32_t g_per_w, int64_t n_states,
                                      const SdpStateDesc* desc, const double* staging, int64_t n_tiles,
                                      const int64_t* tile_off, const int64_t* tile_g_off,
                                      const int32_t* tile_U, int32_t max_tile_U, int32_t* cell,
                                      double* lam, int64_t lam_plane, double* g, void* stream) {
    GridT<double> G;
    int rc = make_grid<double>(grid, &G, nullptr);
    if (rc) return rc;
    if (W < 1 || n_states < 0 || n_tiles < 0 || max_tile_U < 0 || n_states > 32 * n_tiles)
        return fail(SDP_EINVAL, "%s", "sdp_build_tables_tiled: bad sizes");
    if (n_states == 0 || max_tile_U == 0) return SDP_OK;
    if (!desc || !staging || !tile_off || !tile_g_off || !tile_U || !cell || !lam || !g)
        return fail(SDP_EINVAL, "%s", "sdp_build_tables_tiled: NULL pointer");
    int64_t per_tile = (int64_t)W * max_tile_U * 32;
    int bpt = (int)((per_tile + 255) / 256);
    int64_t blocks = n_tiles * bpt;
    if (blocks > 0x7fffffffLL) return fail(SDP_EINVAL, "%s", "sdp_build_tables_tiled: chunk too large");
    cudaStream_t st = (cudaStream_t)stream;
    switch (grid->d) {
        case 1: k_build_tables_tiled<1><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, bpt, n_states, desc, staging, tile_off, tile_g_off, tile_U, cell, lam, lam_plane, g); break;
        case 2: k_build_tables_tiled<2><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, bpt, n_states, desc, staging, tile_off, tile_g_off, tile_U, cell, lam, lam_plane, g); break;
        case 3: k_build_tables_tiled<3><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, bpt, n_states, desc, staging, tile_off, tile_g_off, tile_U, cell, lam, lam_plane, g); break;
        default: k_build_tables_tiled<4><<<(unsigned)blocks, 256, 0, st>>>(G, W, g_per_w, bpt, n_states, desc, staging, tile_off, tile_g_off, tile_U, cell, lam, lam_plane, g); break;
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}


// Factored layouts: the (x,u) part and the (x,w) part of the same expansion.
// Coordinate k of a u entry is read at w index 0, of a w entry at flat control
// index 0 (the host has checked that the staged arrays do not depend on the
// other index), so every value is one the dense build would also have produced.
template <int D>
__device__ __forceinline__ void build_part(const GridT<double>& G, const SdpStateDesc* ds, bool live,
                                           int mask_sel, int u, int w,
                                           const double* __restrict__ staging,
                                           int32_t* __restrict__ cell, double* __restrict__ lam,
                                           int64_t plane, int64_t off) {
    int base = 0, j = 0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        if (!((mask_sel >> k) & 1)) continue;
        double l = 0.0;
        if (live) {
            int q;
            cell_1d<double>(staging[src_offset(ds, k, u, w)], G.smin[k], G.span[k], G.om1[k], G.order[k], q, l);
            base += q * G.stride[k];
        }
        lam[(int64_t)j * plane + off] = l;
        ++j;
    }
    cell[off] = base;
}

template <int D>
__global__ void __launch_bounds__(256)
k_build_factored(GridT<double> G, int W, int u_mask, int tiles_per_state,
                 const SdpStateDesc* __restrict__ desc, const double* __restrict__ staging,
                 int32_t* __restrict__ cell, double* __restrict__ lam, int64_t lam_plane,
                 double* __restrict__ g, int32_t* __restrict__ cell_w, double* __restrict__ lam_w,
                 int64_t lam_w_plane) {
    const int64_t state = blockIdx.x / tiles_per_state;
    const int tile = blockIdx.x % tiles_per_state;
    const SdpStateDesc* ds = desc + state;
    const int e = tile * blockDim.x + threadIdx.x;
    const int w_mask = ~u_mask & ((1 << D) - 1);
    if (e < ds->Upad) {
        const bool live = e < ds->U;
        const int64_t off = ds->entry_off + e;
        build_part<D>(G, ds, live, u_mask, e, 0, staging, cell, lam, lam_plane, off);
        g[off] = live ? staging[src_offset(ds, D, e, 0)] : 0.0;
    } else {
        const int w = e - ds->Upad;
        if (w >= W) return;
        build_part<D>(G, ds, true, w_mask, 0, w, staging, cell_w, lam_w, lam_w_plane, state * W + w);
    }
}

template <int D>
__global__ void __launch_bounds__(256)
k_build_factored_tiled(GridT<double> G, int W, int u_mask, int blocks_per_tile, int64_t n_states,
                       const SdpStateDesc* __restrict__ desc, const double* __restrict__ staging,
                       const int64_t* __restrict__ tile_off, const int32_t* __restrict__ tile_U,
                       int32_t* __restrict__ cell, double* __restrict__ lam, int64_t lam_plane,
                       double* __restrict__ g, int32_t* __restrict__ cell_w,
                       double* __restrict__ lam_w, int64_t lam_w_plane) {
    const int64_t tile = blockIdx.x / blocks_per_tile;
    const int blk = blockIdx.x % blocks_per_tile;
    const int Ut = tile_U[tile];
    const int e = blk * blockDim.x + threadIdx.x;
    if (e >= (Ut + W) * 32) return;
    const int lane = e & 31;
    const int r = e >> 5;
    const int64_t state = tile * 32 + lane;
    const bool in_range = state < n_states;
    const SdpStateDesc* ds = desc + (in_range ? state : 0);
    const int w_mask = ~u_mask & ((1 << D) - 1);
    if (r < Ut) {
        const bool live = in_range && r < ds->U;
        const int64_t off = tile_off[tile] + e;
        build_part<D>(G, ds, live, u_mask, r, 0, staging, cell, lam, lam_plane, off);
        g[off] = live ? staging[src_offset(ds, D, r, 0)] : 0.0;
    } else {
        const int w = r - Ut;
        build_part<D>(G, ds, in_range, w_mask, 0, w, staging, cell_w, lam_w, lam_w_plane,
                      (tile * W + w) * 32 + lane);
    }
}

static int check_factored_args(int d, int W, int u_mask, const char* who) {
    const int full = (1 << d) - 1;
    if (d < 2 || d > 3) return fail(SDP_EINVAL, "%s: factored tables need 2 or 3 state variables", who);
    if (W < 1 || u_mask <= 0 || u_mask >= full)
        return fail(SDP_EINVAL, "%s: u_mask must select at least one and not all coordinates", who);
    return SDP_OK;
}

extern "C" int sdp_build_tables_factored(const SdpGrid* grid, int32_t W, int32_t u_mask, int64_t n_states,
                                         const SdpStateDesc* desc, const double* staging, int32_t* cell,
                                         double* lam, int64_t lam_plane, double* g, int32_t max_Upad,
                                         int32_t* cell_w, double* lam_w, int64_t lam_w_plane,
                                         void* stream) {
    GridT<double> G;
    int rc = make_grid<double>(grid, &G, nullptr);
    if (rc) return rc;
    rc = check_factored_args(grid->d, W, u_mask, "sdp_build_tables_factored");
    if (rc) return rc;
    if (n_states < 0 || max_Upad < 0 || (max_Upad & 3))
        return fail(SDP_EINVAL, "%s", "sdp_build_tables_factored: bad sizes");
    if (n_states == 0) return SDP_OK;
    if (!desc || !staging || !cell || !lam || !g || !cell_w || !lam_w)
        return fail(SDP_EINVAL, "%s", "sdp_build_tables_factored: NULL pointer");
    int tiles = (int)(((int64_t)max_Upad + W + 255) / 256);
    int64_t blocks = n_states * tiles;
    if (blocks > 0x7fffffffLL) return fail(SDP_EINVAL, "%s", "sdp_build_tables_factored: chunk too large");
    cudaStream_t st = (cudaStream_t)stream;
    if (grid->d == 2)
        k_build_factored<2><<<(unsigned)blocks, 256, 0, st>>>(G, W, u_mask, tiles, desc, staging, cell, lam, lam_plane, g, cell_w, lam_w, lam_w_plane);
    else
        k_build_factored<3><<<(unsigned)blocks, 256, 0, st>>>(G, W, u_mask, tiles, desc, staging, cell, lam, lam_plane, g, cell_w, lam_w, lam_w_plane);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

extern "C" int sdp_build_tables_factored_tiled(const SdpGrid* grid, int32_t W, int32_t u_mask,
                                               int64_t n_states, const SdpStateDesc* desc,
                                               const double* staging, int64_t n_tiles,
                                               const int64_t* tile_off, const int32_t* tile_U,
                                               int32_t max_tile_U, int32_t* cell, double* lam,
                                               int64_t lam_plane, double* g, int32_t* cell_w,
                                               double* lam_w, int64_t lam_w_plane, void* stream) {
    GridT<double> G;
    int rc = make_grid<double>(grid, &G, nullptr);
    if (rc) return rc;
    rc = check_factored_args(grid->d, W, u_mask, "sdp_build_tables_factored_tiled");
    if (rc) return rc;
    if (n_states < 0 || n_tiles < 0 || max_tile_U < 0 || n_states > 32 * n_tiles)
        return fail(SDP_EINVAL, "%s", "sdp_build_tables_factored_tiled: bad sizes");
    if (n_states == 0) return SDP_OK;
    if (!desc || !staging || !tile_off || !tile_U || !cell || !lam || !g || !cell_w || !lam_w)
        return fail(SDP_EINVAL, "%s", "sdp_build_tables_factored_tiled: NULL pointer");
    int64_t per_tile = ((int64_t)max_tile_U + W) * 32;
    int bpt = (int)((per_tile + 255) / 256);
    int64_t blocks = n_tiles * bpt;
    if (blocks > 0x7fffffffLL) return fail(SDP_EINVAL, "%s", "sdp_build_tables_factored_tiled: chunk too large");
    cudaStream_t st = (cudaStream_t)stream;
    if (grid->d == 2)
        k_build_factored_tiled<2><<<(unsigned)blocks, 256, 0, st>>>(G, W, u_mask, bpt, n_states, desc, staging, tile_off, tile_U, cell, lam, lam_plane, g, cell_w, lam_w, lam_w_plane);
    else
        k_build_factored_tiled<3><<<(unsigned)blocks, 256, 0, st>>>(G, W, u_mask, bpt, n_states, desc, staging, tile_off, tile_U, cell, lam, lam_plane, g, cell_w, lam_w, lam_w_plane);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K1: Bellman sweep
// ---------------------------------------------------------------------------
// numpy argmin order on (value, flat index): NaN beats everything, then the
// smaller value, then the smaller index (first minimum wins; stodynprog.py:686,
// SURVEY.md App. A.4).  Returns true when a is strictly preferred over b.
__device__ __forceinline__ bool better(double av, int ai, double bv, int bi) {
    const bool an = (av != av), bn = (bv != bv);
    if (an | bn) return (an & bn) ? (ai < bi) : an;
    if (av < bv) return true;
    if (av > bv) return false;
    return ai < bi;
}

// streamed table fragment for UPL consecutive controls of one (state, w) row
template <int D, int UPL>
struct Frag {
    int cell[UPL];
    double lam[D][UPL];
};

template <int D, int UPL>
__device__ __forceinline__ void load_frag(Frag<D, UPL>& f, const int32_t* __restrict__ cell,
                                          const double* __restrict__ lam, int64_t lam_plane,
                                          int64_t off) {
    if (UPL == 4) {
        int4 c = __ldcs(reinterpret_cast<const int4*>(cell + off));
        f.cell[0] = c.x; f.cell[1] = c.y; f.cell[2] = c.z; f.cell[3] = c.w;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const double2* p = reinterpret_cast<const double2*>(lam + (int64_t)k * lam_plane + off);
            double2 a = __ldcs(p);
            double2 b = __ldcs(p + 1);
            f.lam[k][0] = a.x; f.lam[k][1] = a.y; f.lam[k][2] = b.x; f.lam[k][3] = b.y;
        }
    } else {
        int2 c = __ldcs(reinterpret_cast<const int2*>(cell + off));
        f.cell[0] = c.x; f.cell[1] = c.y;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            double2 a = __ldcs(reinterpret_cast<const double2*>(lam + (int64_t)k * lam_plane + off));
            f.lam[k][0] = a.x; f.lam[k][1] = a.y;
        }
    }
}

template <int UPL>
__device__ __forceinline__ void load_g(double (&gv)[UPL], const double* __restrict__ g, int64_t off) {
    if (UPL == 4) {
        const double2* p = reinterpret_cast<const double2*>(g + off);
        double2 a = __ldcs(p), b = __ldcs(p + 1);
        gv[0] = a.x; gv[1] = a.y; gv[2] = b.x; gv[3] = b.y;
    } else {
        double2 a = __ldcs(reinterpret_cast<const double2*>(g + off));
        gv[0] = a.x; gv[1] = a.y;
    }
}

template <int D, int UPL>
__global__ void __launch_bounds__(256)
k_sweep(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
        double* __restrict__ part_val, int32_t* __restrict__ part_idx) {
    extern __shared__ double p_sh[];
    for (int i = threadIdx.x; i < T.W; i += blockDim.x) p_sh[i] = T.expect ? T.p[i] : 1.0;
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int64_t item_id = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    const int W = T.W;
    const int64_t pitch = it.Upad;

    double best_v = CUDART_INF;
    int best_i = INT_MAX;

    // lane handles controls [u0, u0+UPL) of the run, then strides by 32*UPL
    for (int u0 = lane * UPL; u0 < it.u_count; u0 += 32 * UPL) {
        double acc[UPL];
        double gv[UPL];
#pragma unroll
        for (int j = 0; j < UPL; ++j) acc[j] = 0.0;
        if (!T.g_per_w) load_g<UPL>(gv, T.g, it.g_base + u0);

        Frag<D, UPL> cur, nxt;
        load_frag<D, UPL>(cur, T.cell, T.lam, T.lam_plane, it.entry_base + u0);
        for (int w = 0; w < W; ++w) {
            const int64_t off_next = it.entry_base + (int64_t)(w + 1) * pitch + u0;
            if (w + 1 < W) load_frag<D, UPL>(nxt, T.cell, T.lam, T.lam_plane, off_next);
            if (T.g_per_w) load_g<UPL>(gv, T.g, it.g_base + (int64_t)w * pitch + u0);
            const double pw = p_sh[w];
#pragma unroll
            for (int j = 0; j < UPL; ++j) {
                double lam[D];
#pragma unroll
                for (int k = 0; k < D; ++k) lam[k] = cur.lam[k][j];
                double v = Lerp<double, D, 0>::eval(Jprev, cur.cell[j], G.stride, lam);
                double jg = add_(gv[j], v);            // g + J_next(f(x,u,w))   stodynprog.py:677
                if (T.expect) acc[j] = add_(acc[j], mul_(jg, pw));   // np.inner over w   :682
                else acc[j] = jg;                      // deterministic: J = J_k_grid      :679-680
            }
            if (w + 1 < W) cur = nxt;
        }
#pragma unroll
        for (int j = 0; j < UPL; ++j) {
            const int u = u0 + j;
            if (u < it.u_count) {
                const int idx = it.u_begin + u;
                if (better(acc[j], idx, best_v, best_i)) { best_v = acc[j]; best_i = idx; }
            }
        }
    }
    // lexicographic (value, index) min across the warp
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, best_v, s);
        int oi = __shfl_xor_sync(0xffffffffu, best_i, s);
        if (better(ov, oi, best_v, best_i)) { best_v = ov; best_i = oi; }
    }
    if (lane == 0) {
        part_val[item_id] = best_v;
        part_idx[item_id] = best_i;
    }
}

// combine the partial minima of each state's items (in item order = control order)
__global__ void __launch_bounds__(256)
k_sweep_finalize(int64_t n_states, const int64_t* __restrict__ item_begin,
                 const double* __restrict__ part_val, const int32_t* __restrict__ part_idx,
                 double* __restrict__ J_out, int32_t* __restrict__ argmin_out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_states) return;
    int64_t b = item_begin[i], e = item_begin[i + 1];
    double bv = CUDART_INF;
    int bi = INT_MAX;
    for (int64_t k = b; k < e; ++k) {
        double v = part_val[k];
        int ix = part_idx[k];
        if (better(v, ix, bv, bi)) { bv = v; bi = ix; }
    }
    J_out[i] = bv;
    argmin_out[i] = bi;
}

// Layout B: lane <-> state of a 32-state tile; each lane walks the run of
// controls serially (so its running minimum needs no index compare beyond the
// NaN rule), the perturbation loop is batched WB nodes at a time to keep WB
// independent table loads + gathers in flight per lane.
template <int D, int WB>
__global__ void __launch_bounds__(256)
k_sweep_tiled(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
              double* __restrict__ part_val, int32_t* __restrict__ part_idx) {
    extern __shared__ double p_sh[];
    for (int i = threadIdx.x; i < T.W; i += blockDim.x) p_sh[i] = T.expect ? T.p[i] : 1.0;
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int64_t item_id = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    const int W = T.W;
    const int64_t state = (int64_t)it.state * 32 + lane;
    const int Us = (state < T.n_states) ? T.U[state] : 0;

    double best_v = CUDART_INF;
    int best_i = INT_MAX;
    const int32_t* __restrict__ cellp = T.cell + it.entry_base + lane;
    const double* __restrict__ lamp = T.lam + it.entry_base + lane;
    const double* __restrict__ gp = T.g + it.g_base + lane;

    for (int uu = 0; uu < it.u_count; ++uu) {
        const int64_t row = (int64_t)uu * W * 32;
        double acc = 0.0;
        double gv = 0.0;
        if (!T.g_per_w) gv = __ldcs(gp + (int64_t)uu * 32);
        int w = 0;
        for (; w + WB <= W; w += WB) {
            int c[WB];
            double l[WB][D];
            double gw[WB];
#pragma unroll
            for (int b = 0; b < WB; ++b) {
                const int64_t o = row + (int64_t)(w + b) * 32;
                c[b] = __ldcs(cellp + o);
#pragma unroll
                for (int k = 0; k < D; ++k) l[b][k] = __ldcs(lamp + (int64_t)k * T.lam_plane + o);
                gw[b] = T.g_per_w ? __ldcs(gp + o) : gv;
            }
            double v[WB];
#pragma unroll
            for (int b = 0; b < WB; ++b) v[b] = Lerp<double, D, 0>::eval(Jprev, c[b], G.stride, l[b]);
#pragma unroll
            for (int b = 0; b < WB; ++b) {
                double jg = add_(gw[b], v[b]);
                if (T.expect) acc = add_(acc, mul_(jg, p_sh[w + b]));
                else acc = jg;
            }
        }
        for (; w < W; ++w) {
            const int64_t o = row + (int64_t)w * 32;
            int c = __ldcs(cellp + o);
            double l[D];
#pragma unroll
            for (int k = 0; k < D; ++k) l[k] = __ldcs(lamp + (int64_t)k * T.lam_plane + o);
            double gw = T.g_per_w ? __ldcs(gp + o) : gv;
            double jg = add_(gw, Lerp<double, D, 0>::eval(Jprev, c, G.stride, l));
            if (T.expect) acc = add_(acc, mul_(jg, p_sh[w]));
            else acc = jg;
        }
        const int u = it.u_begin + uu;
        if (u < Us && better(acc, u, best_v, best_i)) { best_v = acc; best_i = u; }
    }
    part_val[item_id * 32 + lane] = best_v;
    part_idx[item_id * 32 + lane] = best_i;
}

// ---------------------------------------------------------------------------
// Layout B, software-pipelined variant (default).  ncu on the straight LDG
// kernel shows a pure latency problem (long-scoreboard stalls, L1/L2/DRAM all
// below 65 % busy): the chain "table row -> corner gathers -> arithmetic" is
// serial per warp.  Here the rows of an item (row = one (u,w) pair for the 32
// states of the tile, contiguous in memory) are walked in groups of RB; the
// streaming loads of group i+1 are issued before the 2^d*RB gathers of group i
// are consumed, so every warp keeps RB rows of table traffic and RB rows of
// gathers in flight at all times.
// ---------------------------------------------------------------------------
// running state of one lane (= one state of the tile) while it walks the rows
// (u,w) of its item in order: expectation accumulator over w, minimum over u
struct LaneWalk {
    double best_v, acc, gv, gv_next;
    int best_i, w, uu;
};

__device__ __forceinline__ void walk_row(LaneWalk& s, double jg, double pw, int expect, int W,
                                         int u_begin, int u_count, int Us, bool g_per_w,
                                         const double* __restrict__ gp) {
    if (expect) s.acc = add_(s.acc, mul_(jg, pw));   // np.inner over w   stodynprog.py:682
    else s.acc = jg;                                 // deterministic     :679-680
    if (++s.w == W) {
        const int u = u_begin + s.uu;
        if (u < Us && better(s.acc, u, s.best_v, s.best_i)) { s.best_v = s.acc; s.best_i = u; }
        s.w = 0;
        s.acc = 0.0;
        ++s.uu;
        if (!g_per_w) {
            s.gv = s.gv_next;
            if (s.uu + 1 < u_count) s.gv_next = __ldcs(gp + (int64_t)(s.uu + 1) * 32);
        }
    }
}

template <int D, int RB>
struct RowGroup {
    int c[RB];
    double l[RB][D];
    double gw[RB];
};

// unguarded: all RB rows exist (keeps ptxas free to batch the loads)
template <int D, int RB>
__device__ __forceinline__ void load_rows(RowGroup<D, RB>& g, const int32_t* __restrict__ cellp,
                                          const double* __restrict__ lamp, int64_t lam_plane,
                                          const double* __restrict__ gwp, bool g_per_w, int row0) {
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        const int64_t o = (int64_t)(row0 + r) * 32;
        g.c[r] = __ldcs(cellp + o);
#pragma unroll
        for (int k = 0; k < D; ++k) g.l[r][k] = __ldcs(lamp + (int64_t)k * lam_plane + o);
        g.gw[r] = g_per_w ? __ldcs(gwp + o) : 0.0;
    }
}

template <int D, int RB>
__global__ void __launch_bounds__(256, (RB == 2 ? 3 : (RB == 4 ? 2 : 1)))
k_sweep_tiled_pipe(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
                   double* __restrict__ part_val, int32_t* __restrict__ part_idx) {
    extern __shared__ double p_sh[];
    for (int i = threadIdx.x; i < T.W; i += blockDim.x) p_sh[i] = T.expect ? T.p[i] : 1.0;
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int64_t item_id = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    const int W = T.W;
    const bool g_per_w = T.g_per_w != 0;
    const int64_t state = (int64_t)it.state * 32 + lane;
    const int Us = (state < T.n_states) ? T.U[state] : 0;
    const int n_rows = it.u_count * W;
    const int32_t* __restrict__ cellp = T.cell + it.entry_base + lane;
    const double* __restrict__ lamp = T.lam + it.entry_base + lane;
    const double* __restrict__ gp = T.g + it.g_base + lane;   // g rows: per u, or per (u,w)

    LaneWalk s;
    s.best_v = CUDART_INF; s.best_i = INT_MAX; s.acc = 0.0; s.w = 0; s.uu = 0;
    s.gv = 0.0; s.gv_next = 0.0;
    if (!g_per_w) {
        s.gv = __ldcs(gp);
        if (it.u_count > 1) s.gv_next = __ldcs(gp + 32);
    }

    const int n_full = n_rows / RB;
    RowGroup<D, RB> cur, nxt;
    if (n_full > 0) load_rows<D, RB>(cur, cellp, lamp, T.lam_plane, gp, g_per_w, 0);
    for (int gi = 0; gi < n_full; ++gi) {
        if (gi + 1 < n_full) load_rows<D, RB>(nxt, cellp, lamp, T.lam_plane, gp, g_per_w, (gi + 1) * RB);
        double v[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) v[r] = Lerp<double, D, 0>::eval(Jprev, cur.c[r], G.stride, cur.l[r]);
#pragma unroll
        for (int r = 0; r < RB; ++r)
            walk_row(s, add_(g_per_w ? cur.gw[r] : s.gv, v[r]), p_sh[s.w], T.expect, W, it.u_begin,
                     it.u_count, Us, g_per_w, gp);
        cur = nxt;
    }
    for (int row = n_full * RB; row < n_rows; ++row) {          // tail rows
        RowGroup<D, 1> t;
        load_rows<D, 1>(t, cellp, lamp, T.lam_plane, gp, g_per_w, row);
        const double v = Lerp<double, D, 0>::eval(Jprev, t.c[0], G.stride, t.l[0]);
        walk_row(s, add_(g_per_w ? t.gw[0] : s.gv, v), p_sh[s.w], T.expect, W, it.u_begin, it.u_count,
                 Us, g_per_w, gp);
    }
    part_val[item_id * 32 + lane] = s.best_v;
    part_idx[item_id * 32 + lane] = s.best_i;
}

// ---------------------------------------------------------------------------
// Layout B, TMA-fed variant.  The table region of an item (tile x run of
// controls) is one contiguous run of rows per plane (row = 32 lanes), so each
// warp streams it through its own shared-memory ring with 1-D bulk async copies
// (cp.async.bulk, the TMA engine; SASS UBLKCP) completing on mbarriers: the
// HBM stream never touches the L1/LSU path, which is left to the 2^d-corner
// gathers of J, and the prefetch depth is set by the ring, not by occupancy.
// One elected lane re-arms a slot as soon as the warp has pulled its rows
// into registers.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n.reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

#ifndef SDP_TMA_THREADS
#define SDP_TMA_THREADS 256   // __launch_bounds__ of the TMA kernel (it is launched with NW*32 <= 256 threads)
#endif
#ifndef SDP_TMA_MINB
#define SDP_TMA_MINB 1
#endif
template <int D, int R>
__global__ void __launch_bounds__(SDP_TMA_THREADS, SDP_TMA_MINB)
k_sweep_tiled_tma(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
                  double* __restrict__ part_val, int32_t* __restrict__ part_idx, int S) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int W = T.W;
    const int nw = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int planes = D + (T.g_per_w ? 1 : 0);
    const int stage_bytes = R * 128 + planes * R * 256;
    const int p_bytes = (W * 8 + 127) & ~127;

    double* p_sh = reinterpret_cast<double*>(smem_raw);
    for (int i = threadIdx.x; i < W; i += blockDim.x) p_sh[i] = T.expect ? T.p[i] : 1.0;
    unsigned char* ring = smem_raw + p_bytes + (size_t)warp * S * stage_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + p_bytes + (size_t)nw * S * stage_bytes) + warp * S;
    if (lane == 0) {
        for (int i = 0; i < S; ++i) mbar_init(smem_u32(bars + i), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int64_t item_id = (int64_t)blockIdx.x * nw + warp;
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    const int64_t state = (int64_t)it.state * 32 + lane;
    const int Us = (state < T.n_states) ? T.U[state] : 0;
    const int n_rows = it.u_count * W;
    const int n_stages = (n_rows + R - 1) / R;
    const int32_t* gcell = T.cell + it.entry_base;
    const double* glam = T.lam + it.entry_base;
    const double* ggw = T.g + it.g_base;      // used as a streamed plane when g_per_w

    auto issue = [&](int s) {
        const int slot = s % S;
        const int rows = min(R, n_rows - s * R);
        const uint32_t bar = smem_u32(bars + slot);
        unsigned char* dst = ring + (size_t)slot * stage_bytes;
        mbar_expect_tx(bar, (uint32_t)(rows * (128 + planes * 256)));
        const int64_t e0 = (int64_t)s * R * 32;
        bulk_g2s(smem_u32(dst), gcell + e0, (uint32_t)(rows * 128), bar);
#pragma unroll
        for (int k = 0; k < D; ++k)
            bulk_g2s(smem_u32(dst + R * 128 + k * R * 256), glam + (int64_t)k * T.lam_plane + e0,
                     (uint32_t)(rows * 256), bar);
        if (T.g_per_w)
            bulk_g2s(smem_u32(dst + R * 128 + D * R * 256), ggw + e0, (uint32_t)(rows * 256), bar);
    };

    if (lane == 0) {
        const int pre = min(S, n_stages);
        for (int s = 0; s < pre; ++s) issue(s);
    }

    const bool g_per_w = T.g_per_w != 0;
    const double* __restrict__ gp = T.g + it.g_base + lane;
    LaneWalk ws;
    ws.best_v = CUDART_INF; ws.best_i = INT_MAX; ws.acc = 0.0; ws.w = 0; ws.uu = 0;
    ws.gv = 0.0; ws.gv_next = 0.0;
    if (!g_per_w) {
        ws.gv = __ldcs(gp);
        if (it.u_count > 1) ws.gv_next = __ldcs(gp + 32);
    }

    for (int s = 0; s < n_stages; ++s) {
        const int slot = s % S;
        const int rows = min(R, n_rows - s * R);
        mbar_wait(smem_u32(bars + slot), (uint32_t)((s / S) & 1));
        const unsigned char* st = ring + (size_t)slot * stage_bytes;
        const int32_t* cs = reinterpret_cast<const int32_t*>(st) + lane;
        const double* ls = reinterpret_cast<const double*>(st + R * 128) + lane;
        if (rows == R) {                     // full stage: no per-row guards
            int c[R];
            double l[R][D];
            double gw[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                c[r] = cs[r * 32];
#pragma unroll
                for (int k = 0; k < D; ++k) l[r][k] = ls[k * R * 32 + r * 32];
                gw[r] = g_per_w ? ls[D * R * 32 + r * 32] : 0.0;
            }
            __syncwarp();                    // every lane has pulled its rows out of the slot
            if (lane == 0 && s + S < n_stages) issue(s + S);
            double v[R];
#pragma unroll
            for (int r = 0; r < R; ++r) v[r] = Lerp<double, D, 0>::eval(Jprev, c[r], G.stride, l[r]);
#pragma unroll
            for (int r = 0; r < R; ++r)
                walk_row(ws, add_(g_per_w ? gw[r] : ws.gv, v[r]), p_sh[ws.w], T.expect, W, it.u_begin,
                         it.u_count, Us, g_per_w, gp);
        } else {                             // last, partial stage
            for (int r = 0; r < rows; ++r) {
                const int c = cs[r * 32];
                double l[D];
#pragma unroll
                for (int k = 0; k < D; ++k) l[k] = ls[k * R * 32 + r * 32];
                const double gw = g_per_w ? ls[D * R * 32 + r * 32] : ws.gv;
                const double v = Lerp<double, D, 0>::eval(Jprev, c, G.stride, l);
                walk_row(ws, add_(gw, v), p_sh[ws.w], T.expect, W, it.u_begin, it.u_count, Us,
                         g_per_w, gp);
            }
        }
    }
    part_val[item_id * 32 + lane] = ws.best_v;
    part_idx[item_id * 32 + lane] = ws.best_i;
}

// (tile, lane) holding local state i: 32 consecutive states per tile (layouts B / BF), or -
// layout CF, n_cols > 0 - state i = row*n_cols + col sits in lane row%32 of tile
// col*tiles_per_col + row/32
__device__ __forceinline__ void tile_of_state(int64_t i, int n_cols, int tiles_per_col,
                                              int64_t& tile, int& lane) {
    if (n_cols > 0) {
        const int64_t row = i / n_cols;
        const int col = (int)(i - row * n_cols);
        tile = (int64_t)col * tiles_per_col + (row >> 5);
        lane = (int)(row & 31);
    } else {
        tile = i >> 5;
        lane = (int)(i & 31);
    }
}

__global__ void __launch_bounds__(256)
k_sweep_finalize_tiled(int64_t n_states, const int64_t* __restrict__ item_begin,
                       const double* __restrict__ part_val, const int32_t* __restrict__ part_idx,
                       double* __restrict__ J_out, int32_t* __restrict__ argmin_out,
                       int n_cols, int tiles_per_col) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_states) return;
    int64_t tile;
    int lane;
    tile_of_state(i, n_cols, tiles_per_col, tile, lane);
    int64_t b = item_begin[tile], e = item_begin[tile + 1];
    double bv = CUDART_INF;
    int bi = INT_MAX;
    for (int64_t k = b; k < e; ++k) {
        double v = part_val[k * 32 + lane];
        int ix = part_idx[k * 32 + lane];
        if (better(v, ix, bv, bi)) { bv = v; bi = ix; }
    }
    J_out[i] = bv;
    argmin_out[i] = bi;
}

// ---------------------------------------------------------------------------
// launch tuning.  Defaults come from the environment (SDP_UPL, SDP_WB,
// SDP_TILED_IMPL=tma|ldg, SDP_TMA_R, SDP_TMA_S, SDP_TMA_NW) and can be changed
// at run time through sdp_set_option() (developer tuning sweeps).
// ---------------------------------------------------------------------------
struct Tuning {
    int upl;      // layout A: controls per lane per iteration (2|4)
    int wb;       // layout B, LDG kernel: perturbation nodes batched (1|2|3|5)
    int tma;      // layout B: 0 = straight LDG kernel, 1 = TMA-fed kernel, 2 = software-pipelined LDG kernel
    int rb;       // layout B, pipelined kernel: rows per group (2|4|8)
    int R, S, NW; // TMA ring: rows per stage (4|8), stages, warps per CTA
    int hoist;    // layout AF, u_mask == 1: tabulate the inner interpolation per item (1) or not (0)
    int hoist_upl; // controls per lane per iteration of the hoisted kernel (2|4)
    int p2p_timeout_s; // bound of the peer-flag waits (seconds) before the kernel traps
    int hoist_const;   // layout AF hoisted kernel: constant-W variant for W <= 9 (1) or the runtime-W kernel (0)
    int col_threads;   // layout CF: threads per CTA (one CTA per SM: the column table fills shared memory)
    int col_ub;        // layout CF: controls per lane per iteration (1|2)
    int col_pf;        // layout CF: groups of col_ub controls in flight per lane (1|2)
    int col_dynamic;   // layout CF: warps take the items of a column first come first served (1) or round-robin (0)
    int col_prepass;   // layout CF: column tables from the coalesced pre-pass, copied by vector loads (1) or by the TMA engine (2); 0: gathered by every CTA
    int col_prune;     // layout CF with SdpTables.col_bound: skip the controls that provably lose (1) or evaluate all (0)
    int col_prune_stats; // layout CF pruning sweep: count warp steps and skipped ones (measurements only)
    int pdl;           // programmatic dependent launch of pre-pass / column sweep / combine (1) or plain launches (0)
    int small_combine; // sdp_sweep_finalize_cols: the 128-thread combine that fits next to a streaming CTA (1) or the 1024-thread one (0)
    int carveout;      // layout CF: streaming kernel and small combine ask for the largest shared-memory carve-out (1) or leave it to the driver (0)
    int chain_threads; // sdp_chain_sample: threads per CTA (0 = 256); the results do not depend on it
    int dbg_exchange;  // TIMING EXPERIMENTS ONLY (wrong results): 1 = no stores to remote ranks, 2 = no system fence, 4 = relaxed flag stores
};
static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
static int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}
static Tuning& tuning() {
    static Tuning t = [] {
        Tuning x;
        x.upl = env_int("SDP_UPL", 4) == 2 ? 2 : 4;
        int wb = env_int("SDP_WB", 1);
        x.wb = (wb == 2 || wb == 3 || wb == 5) ? wb : 1;
        // measured on B200 (profiles/): the tiled sweep is bound by L1 wavefronts
        // of the corner gathers, not by the HBM stream, and the LDG kernel's higher
        // occupancy hides the gather latency better than the TMA ring does
        // measured on B200, config #5 (profiles/r1_tuning_tiled_kernels.txt): TMA ring
        // R=8,S=2,NW=4 85.6 % of the HBM roofline, straight LDG 78 %, pipelined LDG 71 %
        const char* impl = getenv("SDP_TILED_IMPL");
        x.tma = 1;
        if (impl && strcmp(impl, "pipe") == 0) x.tma = 2;
        if (impl && strcmp(impl, "ldg") == 0) x.tma = 0;
        int rb = env_int("SDP_RB", 4);
        x.rb = (rb == 2 || rb == 8) ? rb : 4;
        x.R = env_int("SDP_TMA_R", 8) == 4 ? 4 : 8;
        x.S = env_int("SDP_TMA_S", 2);
        x.NW = env_int("SDP_TMA_NW", 4);
        x.hoist = env_int("SDP_HOIST", 1) != 0;
        x.hoist_upl = env_int("SDP_HOIST_UPL", 2) == 4 ? 4 : 2;
        x.p2p_timeout_s = clampi(env_int("SDP_P2P_TIMEOUT_S", 600), 1, 86400);
        x.hoist_const = env_int("SDP_HOIST_CONST", 1) != 0;
        // measured on config #5 (profiles/r1_column_tuning.txt): 512 threads 1.30 ms per sweep,
        // 640 (5 warps per scheduler, 96 registers) 1.24 ms, 704 1.38 ms, 768 1.22-1.26 ms
        // round 2 (profiles/r2_emu_variants.txt, one band / one shard of eight): 640 threads round-robin
        // 1.180 / 0.1788 ms, 640 first-come-first-served 1.168 / 0.1729, 768 round-robin 1.158 / 0.1746,
        // 768 first-come-first-served 1.148 / 0.1726 -> 768 threads, items handed out dynamically
        // 0 = by kernel: 768, or 640 for the pruning sweep (column_threads)
        x.col_threads = env_int("SDP_COL_THREADS", 0) ? clampi(env_int("SDP_COL_THREADS", 0), 128, 768) / 32 * 32 : 0;
        x.col_ub = env_int("SDP_COL_UB", 2) == 1 ? 1 : 2;
        x.col_pf = env_int("SDP_COL_PF", 2) == 1 ? 1 : 2;
        x.col_prepass = clampi(env_int("SDP_COL_PREPASS", 3), 0, 3);
        x.col_dynamic = env_int("SDP_COL_DYNAMIC", 1) != 0;
        x.col_prune = env_int("SDP_COL_PRUNE", 1) != 0;
        x.col_prune_stats = 0;
        x.dbg_exchange = 0;
        x.pdl = env_int("SDP_PDL", 1) != 0;
        x.small_combine = env_int("SDP_SMALL_COMBINE", 1) != 0;
        x.carveout = env_int("SDP_CARVEOUT", 1) != 0;
        x.chain_threads = 0;
        return x;
    }();
    return t;
}
extern "C" int sdp_set_option(const char* name, int value) {
    if (!name) return fail(SDP_EINVAL, "%s", "sdp_set_option: NULL name");
    Tuning& t = tuning();
    if (!strcmp(name, "upl")) t.upl = (value == 2) ? 2 : 4;
    else if (!strcmp(name, "wb")) t.wb = (value == 2 || value == 3 || value == 5) ? value : 1;
    else if (!strcmp(name, "tma")) t.tma = clampi(value, 0, 2);
    else if (!strcmp(name, "rb")) t.rb = (value == 2 || value == 8) ? value : 4;
    else if (!strcmp(name, "tma_rows")) t.R = (value == 8) ? 8 : 4;
    else if (!strcmp(name, "tma_stages")) t.S = value;
    else if (!strcmp(name, "tma_warps")) t.NW = value;
    else if (!strcmp(name, "hoist")) t.hoist = value != 0;
    else if (!strcmp(name, "hoist_upl")) t.hoist_upl = (value == 4) ? 4 : 2;
    else if (!strcmp(name, "p2p_timeout_s")) t.p2p_timeout_s = clampi(value, 1, 86400);
    else if (!strcmp(name, "hoist_const")) t.hoist_const = value != 0;
    else if (!strcmp(name, "col_threads")) t.col_threads = value ? clampi(value, 128, 768) / 32 * 32 : 0;
    else if (!strcmp(name, "col_ub")) t.col_ub = (value == 1) ? 1 : 2;
    else if (!strcmp(name, "col_pf")) t.col_pf = (value == 1) ? 1 : 2;
    else if (!strcmp(name, "col_prepass")) t.col_prepass = clampi(value, 0, 3);
    else if (!strcmp(name, "col_dynamic")) t.col_dynamic = value != 0;
    else if (!strcmp(name, "col_prune")) t.col_prune = value != 0;
    else if (!strcmp(name, "col_prune_stats")) t.col_prune_stats = value != 0;
    else if (!strcmp(name, "dbg_exchange")) t.dbg_exchange = value;
    else if (!strcmp(name, "pdl")) t.pdl = value != 0;
    else if (!strcmp(name, "small_combine")) t.small_combine = value != 0;
    else if (!strcmp(name, "chain_threads")) t.chain_threads = value ? clampi(value, 32, 1024) / 32 * 32 : 0;
    else return fail(SDP_EINVAL, "sdp_set_option: unknown option %s", name);
    return SDP_OK;
}

template <int D, int R>
static int launch_tiled_tma(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                            double* part_val, int32_t* part_idx, cudaStream_t st, int S, int NW,
                            bool* launched) {
    const int planes = D + (T.g_per_w ? 1 : 0);
    const size_t stage_bytes = (size_t)R * 128 + (size_t)planes * R * 256;
    const size_t p_bytes = ((size_t)T.W * 8 + 127) & ~(size_t)127;
    size_t shm = p_bytes + (size_t)NW * S * stage_bytes + (size_t)NW * S * 8;
    while (shm > 200 * 1024 && NW > 1) {     // shrink the CTA until the rings fit
        NW >>= 1;
        shm = p_bytes + (size_t)NW * S * stage_bytes + (size_t)NW * S * 8;
    }
    *launched = false;
    if (shm > 200 * 1024) return SDP_OK;     // does not fit: caller falls back to the LDG kernel
    static size_t attr_set[5][9] = {};
    if (attr_set[D][R] < shm) {
        cudaError_t e = cudaFuncSetAttribute(k_sweep_tiled_tma<D, R>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm);
        if (e != cudaSuccess) return fail(SDP_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        attr_set[D][R] = shm;
    }
    unsigned blocks = (unsigned)((T.n_items + NW - 1) / NW);
    k_sweep_tiled_tma<D, R><<<blocks, NW * 32, shm, st>>>(G, T, Jprev, part_val, part_idx, S);
    note_kernel("k_sweep_tiled_tma<%d,%d> [%d stages, %d threads]", D, R, S, NW * 32);
    *launched = true;
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

template <int D>
static int launch_sweep(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                        double* part_val, int32_t* part_idx, cudaStream_t st) {
    const int warps = 8;
    unsigned blocks = (unsigned)((T.n_items + warps - 1) / warps);
    size_t shm = (size_t)T.W * sizeof(double);
    const Tuning t = tuning();
    if (T.layout == SDP_LAYOUT_STATE_MINOR) {
        if (t.tma == 2) {
            switch (t.rb) {
                case 2: k_sweep_tiled_pipe<D, 2><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx); break;
                case 8: k_sweep_tiled_pipe<D, 8><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx); break;
                default: k_sweep_tiled_pipe<D, 4><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx); break;
            }
            note_kernel("k_sweep_tiled_pipe<%d,%d>", D, (t.rb == 2 || t.rb == 8) ? t.rb : 4);
            SDP_LAUNCH_CHECK();
            return SDP_OK;
        }
        if (t.tma == 1) {
            bool launched = false;
            const int S = clampi(t.S, 2, 16), NW = clampi(t.NW, 1, 8);
            int rc = (t.R == 8)
                ? launch_tiled_tma<D, 8>(G, T, Jprev, part_val, part_idx, st, S, NW, &launched)
                : launch_tiled_tma<D, 4>(G, T, Jprev, part_val, part_idx, st, S, NW, &launched);
            if (rc || launched) return rc;
        }
        switch (t.wb) {
            case 2: k_sweep_tiled<D, 2><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx); break;
            case 3: k_sweep_tiled<D, 3><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx); break;
            case 5: k_sweep_tiled<D, 5><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx); break;
            default: k_sweep_tiled<D, 1><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx); break;
        }
        note_kernel("k_sweep_tiled<%d,%d>", D, (t.wb == 2 || t.wb == 3 || t.wb == 5) ? t.wb : 1);
    } else if (t.upl == 2) {
        k_sweep<D, 2><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx);
        note_kernel("k_sweep<%d,2>", D);
    } else {
        k_sweep<D, 4><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx);
        note_kernel("k_sweep<%d,4>", D);
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}


// ---------------------------------------------------------------------------
// Factored sweeps (layouts AF / BF): cell = cell_u + cell_w, the weight vector
// is merged from the u-part and the w-part in coordinate order, so the nested
// lerp sees exactly the operands the dense tables would have held.
// ---------------------------------------------------------------------------
template <int D, int MASK>
struct Fact {
    static constexpr int NU = ((MASK >> 0) & 1) + ((MASK >> 1) & 1) + ((MASK >> 2) & 1) + ((MASK >> 3) & 1);
    static constexpr int NW = D - NU;
    __device__ __forceinline__ static void merge(double (&lam)[D], const double (&lu)[NU], const double (&lw)[NW]) {
        int ju = 0, jw = 0;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            if ((MASK >> k) & 1) lam[k] = lu[ju++];
            else lam[k] = lw[jw++];
        }
    }
};

// probabilities as launch constants (kernel parameter = constant bank, operands of the
// DMULs themselves; see k_sweep_fact_tiled and k_sweep_fact_hoist_c)
struct PVals {
    double v[SDP_FACTORED_MAX_W_REG];
};

// AF: one warp per run of controls of one state, lane <-> UPL consecutive
// controls; the state's w-part (W entries, warp-uniform) sits in shared memory.
template <int D, int MASK, int UPL>
__global__ void __launch_bounds__(256)
k_sweep_fact(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
             double* __restrict__ part_val, int32_t* __restrict__ part_idx) {
    constexpr int NU = Fact<D, MASK>::NU, NW = Fact<D, MASK>::NW;
    extern __shared__ __align__(16) unsigned char fsm[];
    const int W = T.W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    double* p_sh = reinterpret_cast<double*>(fsm);
    double* lw_sh = p_sh + W + (size_t)warp * NW * W;                       // [NW][W] of this warp
    int* cw_sh = reinterpret_cast<int*>(p_sh + W + (size_t)nwarps * NW * W) + warp * W;
    for (int i = threadIdx.x; i < W; i += blockDim.x) p_sh[i] = T.expect ? T.p[i] : 1.0;
    __syncthreads();

    const int64_t item_id = (int64_t)blockIdx.x * nwarps + warp;
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    for (int w = lane; w < W; w += 32) {
        const int64_t f = (int64_t)it.state * W + w;
        cw_sh[w] = __ldg(T.cell_w + f);
#pragma unroll
        for (int j = 0; j < NW; ++j) lw_sh[j * W + w] = __ldg(T.lam_w + (int64_t)j * T.lam_w_plane + f);
    }
    __syncwarp();

    double best_v = CUDART_INF;
    int best_i = INT_MAX;
    for (int u0 = lane * UPL; u0 < it.u_count; u0 += 32 * UPL) {
        const int64_t off = it.entry_base + u0;
        int cu[UPL];
        double lu[UPL][NU], gv[UPL], acc[UPL];
        {
            Frag<NU, UPL> f;
            load_frag<NU, UPL>(f, T.cell, T.lam, T.lam_plane, off);
            load_g<UPL>(gv, T.g, off);
#pragma unroll
            for (int j = 0; j < UPL; ++j) {
                cu[j] = f.cell[j];
                acc[j] = 0.0;
#pragma unroll
                for (int k = 0; k < NU; ++k) lu[j][k] = f.lam[k][j];
            }
        }
#pragma unroll 3
        for (int w = 0; w < W; ++w) {
            const int cw = cw_sh[w];
            const double pw = p_sh[w];
            double lw[NW];
#pragma unroll
            for (int k = 0; k < NW; ++k) lw[k] = lw_sh[k * W + w];
#pragma unroll
            for (int j = 0; j < UPL; ++j) {
                double lam[D];
                Fact<D, MASK>::merge(lam, lu[j], lw);
                const double v = Lerp<double, D, 0>::eval(Jprev, cu[j] + cw, G.stride, lam);
                const double jg = add_(gv[j], v);
                if (T.expect) acc[j] = add_(acc[j], mul_(jg, pw));
                else acc[j] = jg;
            }
        }
#pragma unroll
        for (int j = 0; j < UPL; ++j) {
            const int u = u0 + j;
            if (u < it.u_count) {
                const int idx = it.u_begin + u;
                if (better(acc[j], idx, best_v, best_i)) { best_v = acc[j]; best_i = idx; }
            }
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, best_v, s);
        int oi = __shfl_xor_sync(0xffffffffu, best_i, s);
        if (better(ov, oi, best_v, best_i)) { best_v = ov; best_i = oi; }
    }
    if (lane == 0) {
        part_val[item_id] = best_v;
        part_idx[item_id] = best_i;
    }
}

// BF: lane <-> state of a 32-state tile; the lane's w-part (W <= WM <= 9 entries)
// lives in registers, the u-part is streamed one control ahead.  The w loop is
// fully unrolled over WM slots with NO guard on the gathers (slots >= W repeat
// slot W-1, so they hit the same lines): ncu on the guarded version showed one
// exposed L1/L2 round trip per perturbation node (the uniform `w < W` branches
// kept the 4*W corner loads of a control from being issued together).
// AF with hoisted inner interpolation (u_mask == 1: coordinate 0 follows the
// control, every other coordinate the perturbation - the structure of all the
// reference's storage examples).  The nested lerp is
//     (1-l0)*R(q0, w) + l0*R(q0+1, w),   R(r, w) = lerp over axes 1.. of J[r, ...]
// and R depends on the ROW r and on w only, not on the control.  With a fine
// control grid the controls of an item fall into a handful of rows, so the warp
// first tabulates R for the item's row range in shared memory ((rows+1)*W inner
// lerps, the very operations the reference does, done once instead of once per
// control) and the per-backup work shrinks from 2^d gathers + (2^d-1) lerps to
// two shared-memory reads + one lerp.  Items whose row range does not fit the
// table take the generic path below.  Bit-identical by construction.
template <int D, int UPL>
__global__ void __launch_bounds__(256)
k_sweep_fact_hoist(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
                   double* __restrict__ part_val, int32_t* __restrict__ part_idx, int RP,
                   double inv_stride0) {
    constexpr int NW = D - 1;
    extern __shared__ __align__(16) unsigned char fsm[];
    const int W = T.W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    // layout: p[W] | per warp: R[W][RP+1], lw[NW][W] | per warp: cw[W]
    double* p_sh = reinterpret_cast<double*>(fsm);
    const int per_warp_d = W * (RP + 1) + NW * W;
    double* R_sh = p_sh + W + (size_t)warp * per_warp_d;
    double* lw_sh = R_sh + W * (RP + 1);
    int* cw_sh = reinterpret_cast<int*>(p_sh + W + (size_t)nwarps * per_warp_d) + warp * W;
    for (int i = threadIdx.x; i < W; i += blockDim.x) p_sh[i] = T.expect ? T.p[i] : 1.0;
    __syncthreads();

    const int64_t item_id = (int64_t)blockIdx.x * nwarps + warp;
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    for (int w = lane; w < W; w += 32) {
        const int64_t f = (int64_t)it.state * W + w;
        cw_sh[w] = __ldg(T.cell_w + f);
#pragma unroll
        for (int j = 0; j < NW; ++j) lw_sh[j * W + w] = __ldg(T.lam_w + (int64_t)j * T.lam_w_plane + f);
    }
    // row range of the item's controls (cell_u = q0 * stride0)
    int cmin = INT_MAX, cmax = INT_MIN;
    for (int u0 = lane * 4; u0 < it.u_count; u0 += 128) {
        const int4 c = *reinterpret_cast<const int4*>(T.cell + it.entry_base + u0);
        const int cc[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (u0 + j < it.u_count) { cmin = min(cmin, cc[j]); cmax = max(cmax, cc[j]); }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, s));
        cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, s));
    }
    const int stride0 = G.stride[0];
    const int r0 = cmin / stride0;
    const int nrows = cmax / stride0 - r0 + 1;       // rows r0 .. r0+nrows-1, plus the upper corner row
    const bool hoist = nrows <= RP;
    __syncwarp();
    // The u-part is streamed one fragment ahead (ncu: 28 % of the stall samples of the
    // single-buffered loop sat on the first use of the streamed cell); the first
    // fragment is requested here so that its latency overlaps the table build.
    Frag<1, UPL> f_n;
    double g_n[UPL];
    int u0 = lane * UPL;
    if (u0 < it.u_count) {
        load_frag<1, UPL>(f_n, T.cell, T.lam, T.lam_plane, it.entry_base + u0);
        load_g<UPL>(g_n, T.g, it.entry_base + u0);
    }
    if (hoist) {
        const int RS = RP + 1;
        for (int idx = lane; idx < (nrows + 1) * W; idx += 32) {
            const int r = idx / W, w = idx - r * W;
            double lam[D];
            lam[0] = 0.0;
#pragma unroll
            for (int k = 0; k < NW; ++k) lam[k + 1] = lw_sh[k * W + w];
            R_sh[w * RS + r] = Lerp<double, D, 1>::eval(Jprev, (r0 + r) * stride0 + cw_sh[w], G.stride, lam);
        }
        __syncwarp();
    }

    double best_v = CUDART_INF;
    int best_i = INT_MAX;
    for (; u0 < it.u_count; u0 += 32 * UPL) {
        int cu[UPL];
        double lu[UPL], gv[UPL], acc[UPL];
#pragma unroll
        for (int j = 0; j < UPL; ++j) { cu[j] = f_n.cell[j]; lu[j] = f_n.lam[0][j]; gv[j] = g_n[j]; acc[j] = 0.0; }
        if (u0 + 32 * UPL < it.u_count) {
            const int64_t off_n = it.entry_base + u0 + 32 * UPL;
            load_frag<1, UPL>(f_n, T.cell, T.lam, T.lam_plane, off_n);
            load_g<UPL>(g_n, T.g, off_n);
        }
        if (hoist) {
            const int RS = RP + 1;
            int r[UPL];
            double oml[UPL];
#pragma unroll
            for (int j = 0; j < UPL; ++j) {
                // q0 = cu / stride0 exactly (cu is a multiple of stride0 below 2^31)
                int q = __double2int_rn(__dmul_rn((double)cu[j], inv_stride0)) - r0;
                r[j] = max(0, min(q, nrows - 1));     // padding entries (cell 0) stay in range
                oml[j] = sub_(1.0, lu[j]);
            }
#pragma unroll 3
            for (int w = 0; w < W; ++w) {
                const double pw = p_sh[w];
                const double* Rw = R_sh + w * RS;
#pragma unroll
                for (int j = 0; j < UPL; ++j) {
                    const double v = add_(mul_(oml[j], Rw[r[j]]), mul_(lu[j], Rw[r[j] + 1]));
                    const double jg = add_(gv[j], v);
                    if (T.expect) acc[j] = add_(acc[j], mul_(jg, pw));
                    else acc[j] = jg;
                }
            }
        } else {
#pragma unroll 3
            for (int w = 0; w < W; ++w) {
                const int cw = cw_sh[w];
                const double pw = p_sh[w];
                double lam[UPL][D];
#pragma unroll
                for (int j = 0; j < UPL; ++j) {
                    lam[j][0] = lu[j];
#pragma unroll
                    for (int k = 0; k < NW; ++k) lam[j][k + 1] = lw_sh[k * W + w];
                }
#pragma unroll
                for (int j = 0; j < UPL; ++j) {
                    const double v = Lerp<double, D, 0>::eval(Jprev, cu[j] + cw, G.stride, lam[j]);
                    const double jg = add_(gv[j], v);
                    if (T.expect) acc[j] = add_(acc[j], mul_(jg, pw));
                    else acc[j] = jg;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < UPL; ++j) {
            const int u = u0 + j;
            if (u < it.u_count) {
                const int idx = it.u_begin + u;
                if (better(acc[j], idx, best_v, best_i)) { best_v = acc[j]; best_i = idx; }
            }
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, best_v, s);
        int oi = __shfl_xor_sync(0xffffffffu, best_i, s);
        if (better(ov, oi, best_v, best_i)) { best_v = ov; best_i = oi; }
    }
    if (lane == 0) {
        part_val[item_id] = best_v;
        part_idx[item_id] = best_i;
    }
}

// The same hoisted sweep for W <= 9 perturbation nodes (WM = 3 | 5 | 9 unrolled slots).
// ncu on the kernel above: 22 issued instructions per backup for 7 fp64 operations - the
// runtime-W loop recomputes two shared-memory addresses per (control, w), reads p[w]
// from shared memory and carries remainder loops.  Here the table is row-major
// R[row][w] (the W values a control needs from a row are contiguous: one base address
// per control, immediates per w), the w loop is fully unrolled with uniform guards and
// the probabilities are launch constants.  Same operations on the same operands.
template <int D, int WM>
__global__ void __launch_bounds__(256)
k_sweep_fact_hoist_c(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
                     double* __restrict__ part_val, int32_t* __restrict__ part_idx, int RP,
                     double inv_stride0, PVals PV) {
    constexpr int NW = D - 1;
    constexpr int UPL = 2;
    extern __shared__ __align__(16) unsigned char fsm[];
    const int W = T.W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    // per warp: R[RP+1][W], lw[NW][W] | per warp: cw[W]
    const int per_warp_d = W * (RP + 1) + NW * W;
    double* R_sh = reinterpret_cast<double*>(fsm) + (size_t)warp * per_warp_d;
    double* lw_sh = R_sh + W * (RP + 1);
    int* cw_sh = reinterpret_cast<int*>(reinterpret_cast<double*>(fsm) + (size_t)nwarps * per_warp_d) + warp * W;

    const int64_t item_id = (int64_t)blockIdx.x * nwarps + warp;
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    for (int w = lane; w < W; w += 32) {
        const int64_t f = (int64_t)it.state * W + w;
        cw_sh[w] = __ldg(T.cell_w + f);
#pragma unroll
        for (int j = 0; j < NW; ++j) lw_sh[j * W + w] = __ldg(T.lam_w + (int64_t)j * T.lam_w_plane + f);
    }
    // row range of the item's controls (cell_u = q0 * stride0)
    int cmin = INT_MAX, cmax = INT_MIN;
    for (int u = lane * 4; u < it.u_count; u += 128) {
        const int4 c = *reinterpret_cast<const int4*>(T.cell + it.entry_base + u);
        const int cc[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (u + j < it.u_count) { cmin = min(cmin, cc[j]); cmax = max(cmax, cc[j]); }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, s));
        cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, s));
    }
    const int stride0 = G.stride[0];
    const int r0 = cmin / stride0;
    const int nrows = cmax / stride0 - r0 + 1;
    const bool hoist = nrows <= RP;
    __syncwarp();
    Frag<1, UPL> f_n;
    double g_n[UPL];
    int u0 = lane * UPL;
    if (u0 < it.u_count) {
        load_frag<1, UPL>(f_n, T.cell, T.lam, T.lam_plane, it.entry_base + u0);
        load_g<UPL>(g_n, T.g, it.entry_base + u0);
    }
    if (hoist) {
        for (int idx = lane; idx < (nrows + 1) * W; idx += 32) {
            const int r = idx / W, w = idx - r * W;
            double lam[D];
            lam[0] = 0.0;
#pragma unroll
            for (int k = 0; k < NW; ++k) lam[k + 1] = lw_sh[k * W + w];
            R_sh[idx] = Lerp<double, D, 1>::eval(Jprev, (r0 + r) * stride0 + cw_sh[w], G.stride, lam);
        }
        __syncwarp();
    }

    double best_v = CUDART_INF;
    int best_i = INT_MAX;
    for (; u0 < it.u_count; u0 += 32 * UPL) {
        int cu[UPL];
        double lu[UPL], gv[UPL], acc[UPL];
#pragma unroll
        for (int j = 0; j < UPL; ++j) { cu[j] = f_n.cell[j]; lu[j] = f_n.lam[0][j]; gv[j] = g_n[j]; acc[j] = 0.0; }
        if (u0 + 32 * UPL < it.u_count) {
            const int64_t off_n = it.entry_base + u0 + 32 * UPL;
            load_frag<1, UPL>(f_n, T.cell, T.lam, T.lam_plane, off_n);
            load_g<UPL>(g_n, T.g, off_n);
        }
        if (hoist) {
            const double* Ra[UPL];
            const double* Rb[UPL];
            double oml[UPL];
#pragma unroll
            for (int j = 0; j < UPL; ++j) {
                // q0 = cu / stride0 exactly (cu is a multiple of stride0 below 2^31)
                int q = __double2int_rn(__dmul_rn((double)cu[j], inv_stride0)) - r0;
                q = max(0, min(q, nrows - 1));        // padding entries (cell 0) stay in range
                Ra[j] = R_sh + q * W;
                Rb[j] = Ra[j] + W;
                oml[j] = sub_(1.0, lu[j]);
            }
            if (W == WM) {
                // all slots live: no guards, so the 2*UPL*WM shared-memory reads of a
                // control pair are issued together
                double v[UPL][WM];
#pragma unroll
                for (int w = 0; w < WM; ++w)
#pragma unroll
                    for (int j = 0; j < UPL; ++j)
                        v[j][w] = add_(mul_(oml[j], Ra[j][w]), mul_(lu[j], Rb[j][w]));
#pragma unroll
                for (int w = 0; w < WM; ++w)
#pragma unroll
                    for (int j = 0; j < UPL; ++j) {
                        const double jg = add_(gv[j], v[j][w]);
                        if (T.expect) acc[j] = add_(acc[j], mul_(jg, PV.v[w]));
                        else acc[j] = jg;
                    }
            } else {
#pragma unroll
                for (int w = 0; w < WM; ++w) {
                    if (w < W) {
#pragma unroll
                        for (int j = 0; j < UPL; ++j) {
                            const double v = add_(mul_(oml[j], Ra[j][w]), mul_(lu[j], Rb[j][w]));
                            const double jg = add_(gv[j], v);
                            if (T.expect) acc[j] = add_(acc[j], mul_(jg, PV.v[w]));
                            else acc[j] = jg;
                        }
                    }
                }
            }
        } else {
            for (int w = 0; w < W; ++w) {
                const int cw = cw_sh[w];
                const double pw = T.expect ? __ldg(T.p + w) : 1.0;
#pragma unroll
                for (int j = 0; j < UPL; ++j) {
                    double lam[D];
                    lam[0] = lu[j];
#pragma unroll
                    for (int k = 0; k < NW; ++k) lam[k + 1] = lw_sh[k * W + w];
                    const double v = Lerp<double, D, 0>::eval(Jprev, cu[j] + cw, G.stride, lam);
                    const double jg = add_(gv[j], v);
                    if (T.expect) acc[j] = add_(acc[j], mul_(jg, pw));
                    else acc[j] = jg;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < UPL; ++j) {
            const int u = u0 + j;
            if (u < it.u_count) {
                const int idx = it.u_begin + u;
                if (better(acc[j], idx, best_v, best_i)) { best_v = acc[j]; best_i = idx; }
            }
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, best_v, s);
        int oi = __shfl_xor_sync(0xffffffffu, best_i, s);
        if (better(ov, oi, best_v, best_i)) { best_v = ov; best_i = oi; }
    }
    if (lane == 0) {
        part_val[item_id] = best_v;
        part_idx[item_id] = best_i;
    }
}

#ifndef SDP_BF_UB
#define SDP_BF_UB 1      // controls per iteration of the BF kernel
#endif
#ifndef SDP_BF_MINB
#define SDP_BF_MINB 1    // __launch_bounds__ min CTAs per SM of the BF kernel
#endif
// The probabilities enter the BF kernel as launch constants (kernel parameter =
// constant bank, an operand of the DMUL itself): ncu showed the shared-memory
// reads of p[w] taking 1 of the ~9.6 L1 data-pipe wavefronts per warp step of a
// kernel that is bound by exactly that pipe.

template <int D, int MASK, int WM>
__global__ void __launch_bounds__(128, SDP_BF_MINB)
k_sweep_fact_tiled(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
                   double* __restrict__ part_val, int32_t* __restrict__ part_idx, PVals PV) {
    constexpr int NU = Fact<D, MASK>::NU, NW = Fact<D, MASK>::NW;
    constexpr int UB = SDP_BF_UB;

    const int lane = threadIdx.x & 31;
    const int64_t item_id = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item_id >= T.n_items) return;
    const SdpItem it = T.items[item_id];
    const int W = T.W;
    const int64_t state = (int64_t)it.state * 32 + lane;
    const int Us = (state < T.n_states) ? T.U[state] : 0;

    int cw[WM];
    double lw[WM][NW];
#pragma unroll
    for (int w = 0; w < WM; ++w) {
        const int ws = min(w, W - 1);
        const int64_t f = ((int64_t)it.state * W + ws) * 32 + lane;
        cw[w] = __ldg(T.cell_w + f);
#pragma unroll
        for (int k = 0; k < NW; ++k) lw[w][k] = __ldg(T.lam_w + (int64_t)k * T.lam_w_plane + f);
    }

    const int32_t* __restrict__ cup = T.cell + it.entry_base + lane;
    const double* __restrict__ lup = T.lam + it.entry_base + lane;
    const double* __restrict__ gp = T.g + it.g_base + lane;
    double best_v = CUDART_INF;
    int best_i = INT_MAX;
    const int last = it.u_count - 1;

    // group of UB controls, streamed one group ahead (rows past the run repeat its last row)
    int c_n[UB];
    double g_n[UB], l_n[UB][NU];
#pragma unroll
    for (int b = 0; b < UB; ++b) {
        const int64_t o = (int64_t)min(b, last) * 32;
        c_n[b] = __ldcs(cup + o);
        g_n[b] = __ldcs(gp + o);
#pragma unroll
        for (int k = 0; k < NU; ++k) l_n[b][k] = __ldcs(lup + (int64_t)k * T.lam_plane + o);
    }

    for (int uu = 0; uu < it.u_count; uu += UB) {
        int cu[UB];
        double gv[UB], lu[UB][NU];
#pragma unroll
        for (int b = 0; b < UB; ++b) {
            cu[b] = c_n[b];
            gv[b] = g_n[b];
#pragma unroll
            for (int k = 0; k < NU; ++k) lu[b][k] = l_n[b][k];
        }
        if (uu + UB < it.u_count) {
#pragma unroll
            for (int b = 0; b < UB; ++b) {
                const int64_t o = (int64_t)min(uu + UB + b, last) * 32;
                c_n[b] = __ldcs(cup + o);
                g_n[b] = __ldcs(gp + o);
#pragma unroll
                for (int k = 0; k < NU; ++k) l_n[b][k] = __ldcs(lup + (int64_t)k * T.lam_plane + o);
            }
        }
        double v[UB][WM];
#pragma unroll
        for (int b = 0; b < UB; ++b)
#pragma unroll
            for (int w = 0; w < WM; ++w) {
                double lam[D];
                Fact<D, MASK>::merge(lam, lu[b], lw[w]);
                v[b][w] = Lerp<double, D, 0>::eval(Jprev, cu[b] + cw[w], G.stride, lam);
            }
#pragma unroll
        for (int b = 0; b < UB; ++b) {
            double acc = 0.0;
#pragma unroll
            for (int w = 0; w < WM; ++w) {
                const double jg = add_(gv[b], v[b][w]);
                const double nxt = T.expect ? add_(acc, mul_(jg, PV.v[w])) : jg;
                acc = (w < W) ? nxt : acc;        // slots past W do not take part
            }
            const int u = it.u_begin + uu + b;
            if (uu + b <= last && u < Us && better(acc, u, best_v, best_i)) { best_v = acc; best_i = u; }
        }
    }
    part_val[item_id * 32 + lane] = best_v;
    part_idx[item_id * 32 + lane] = best_i;
}

template <int D, int MASK, int WM>
static void launch_fact_tiled_w(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                                double* part_val, int32_t* part_idx, cudaStream_t st) {
    const int warps = 4;
    unsigned blocks = (unsigned)((T.n_items + warps - 1) / warps);
    PVals pv;
    for (int w = 0; w < SDP_FACTORED_MAX_W_REG; ++w)
        pv.v[w] = (w < T.W) ? (T.expect ? T.p_host[w] : 1.0) : 0.0;
    k_sweep_fact_tiled<D, MASK, WM><<<blocks, warps * 32, 0, st>>>(G, T, Jprev, part_val, part_idx, pv);
    note_kernel("k_sweep_fact_tiled<%d,%d,%d>", D, MASK, WM);
}

// ---------------------------------------------------------------------------
// CF: column-shared hoist (include/sdp_b200.h, SDP_LAYOUT_COLUMN_FACTORED).
//
// Layout BF spends 2^d gathers (32 bytes of corner values per lane through the L1
// data pipe) and 2^d-1 lerps on every backup; ncu shows that pipe as its limiter.
// With u_mask == 1 the nested lerp is
//     (1-l0)*R(q0, w) + l0*R(q0+1, w),   R(r, w) = lerp over axes 1.. of J[r, ...]
// and when the (x,w) part of a state does not depend on its axis-0 index (P_next =
// a*P + w does not involve the storage energy), R is the same function of (r, w)
// for ALL states of a column of the grid (fixed indices on the axes 1..d-1).  One
// CTA therefore tabulates R for every row of the grid once per column
// (order[0]*W inner lerps - the very operations every backup of the column would
// repeat) and then sweeps the column's tiles, lane <-> row: a backup is two
// shared-memory reads and one lerp.  Adjacent lanes are adjacent rows, and the row
// pitch is an odd number of doubles (W | 1), so a half-warp's 8-byte reads spread over
// all 32 banks.
//
// Work split: the item list is ordered by tile, i.e. by (band, column); the host cuts
// it into n_segs runs of equal weight, one per CTA (one CTA per SM: the table fills
// shared memory), so a CTA meets few column changes.  Warps take the items of the
// current column round-robin.  Partial minima have the layout of BF.
// ---------------------------------------------------------------------------
// Peer-memory exchange state (see "Multi-GPU" below); declared here because the pre-pass of
// layout CF can start with the flag wait of the previous sweep's exchange.
struct PeersDev {
    int world, rank;
    double* J[SDP_MAX_PEERS];
    int32_t* A[SDP_MAX_PEERS];      // optional: every rank's full-grid argmin buffer (NULL: none)
    unsigned long long* flags[SDP_MAX_PEERS];
    unsigned long long* epoch;
    unsigned int* done;
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// Bounded flag wait: a peer that died (or a call sequence that differs between the
// ranks) must surface as a CUDA error on this rank, not as a hung GPU.
// (default 600 s, like a collective watchdog: the ranks of an SPMD script may reach a
// call minutes apart; `sdp_set_option("p2p_timeout_s", s)` / SDP_P2P_TIMEOUT_S change it)
__device__ __forceinline__ void wait_flag(const unsigned long long* p, unsigned long long e,
                                          unsigned long long timeout_ns) {
    const unsigned long long t0 = global_ns();
    while (ld_acquire_sys(p) < e) {
        __nanosleep(20);
        if (global_ns() - t0 > timeout_ns) __trap();
    }
}

// Pre-pass: the inner-interpolation tables of ALL columns, R[c][r][w] at
// col_table[c*pitch + r*P + w].  A CTA owns a tile of 32 columns x SDP_CT_ROWS rows: it
// computes with lanes along the columns - the w-parts of neighbouring columns point at
// neighbouring cells, so the gathers of a warp are a few lines instead of 32 - into a
// shared-memory tile, then writes each column's run of rows contiguously.
// Programmatic dependent launch (sm_90+): the kernel may be scheduled while its predecessor in the
// stream drains; it calls cudaGridDependencySynchronize() (griddepcontrol.wait) before touching
// anything the predecessor wrote.  Hides the launch latency at the 3 kernel boundaries of a sweep
// (pre-pass -> sweep -> combine), which weighs on the 0.2 ms sweeps of an 8-GPU run.
// tuning().pdl = 0 launches the plain way.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t shm, cudaStream_t st,
                              Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = shm;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = tuning().pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// set by sdp_sweep_partials_after for the duration of the call: the exchange whose flag wait
// the first kernel that reads J_prev must perform (consumed by launch_column_table)
static thread_local const PeersDev* g_wait_peers = nullptr;

// Column pruning (SdpTables.col_bound, DESIGN.md section 4).  With 0 <= l <= 1 and p_w >= 0 the
// value of a control, sum_w p_w*(g + (1-l)*R[q][w] + l*R[q+1][w]), is at least
//     g*sum(p) + m(q),   m(q) = sum_w p_w*min(R[q][w], R[q+1][w]),
// and the value the sweep computes (oml = 1-l, the two products, the add, + g, * p_w, the sum in
// w order, all rounded to nearest, no FMA) lies within (W+4)*u*(|g| + A)*sum(p) of the exact one
// (u = 2^-53, A = max_w max(|R[q][w]|, |R[q+1][w]|)).  Computing m(q), g*sum(p), their sum and
// the subtraction of the margin rounds by at most (W+2)*u*(|g| + A)*sum(p) more, so with W <= 9
// a margin of 32*u*(|g| + A)*sum(p) (24*u needed, the rest covers O(u^2) terms and the rounding
// of the margin itself) plus 2^-1000 (underflow in the products) makes `lb` a lower bound of the
// computed value: lb > best means the control computes a value strictly greater than best, which
// is neither the minimum nor, at a tie, the argmin.  |g| + A <= 2^1000 and p_w <= 1 rule out
// overflow (and NaN) in the computed value; a NaN or inf in R or g fails that test, so such a
// control is never skipped.  Twin: tablebuild.column_prune_skip.
__device__ __forceinline__ double2 column_bound(const double* r, int P, int W, const PVals& PV) {
    double m = 0.0, a = 0.0;
    bool nan = false;
#pragma unroll
    for (int w = 0; w < SDP_FACTORED_MAX_W_REG; ++w) {
        if (w < W) {
            const double x = r[w], y = r[P + w];
            m = add_(m, mul_(PV.v[w], fmin(x, y)));
            a = fmax(a, fmax(fabs(x), fabs(y)));
            nan |= (x != x) | (y != y);
        }
    }
    return make_double2(m, nan ? CUDART_NAN : a);
}
__device__ __forceinline__ bool column_skip(double2 b, double g, double l, double sum_p, double best) {
    const double ga = add_(fabs(g), b.y);
    const double margin = add_(mul_(mul_(ga, sum_p), 0x1p-48), 0x1p-1000);
    const double lb = sub_(add_(mul_(g, sum_p), b.x), margin);
    return (l >= 0.0) & (l <= 1.0) & (ga <= 0x1p1000) & (lb > best);
}

#define SDP_CT_ROWS 16
// `WAIT`: every CTA first waits (lanes 0..world-1, ld.acquire.sys on the local flags) until all
// ranks have published the current epoch, i.e. until the J slabs of the previous sweep have
// landed - the stream-ordered sdp_p2p_wait folded into the first kernel that reads J.
template <int D, bool WAIT>
__global__ void __launch_bounds__(256)
k_column_table(GridT<double> G, SdpTables T, const double* __restrict__ Jprev, int64_t pitch,
               PeersDev PW, unsigned long long timeout_ns, int TR, PVals PV, int bound) {
    constexpr int NW = D - 1;
    extern __shared__ __align__(16) unsigned char tsm[];
    cudaGridDependencySynchronize();       // (programmatic dependent launch: the previous kernel's writes)
    if (WAIT) {
        if (threadIdx.x < PW.world) wait_flag(PW.flags[PW.rank] + threadIdx.x, *PW.epoch, timeout_ns);
        __syncthreads();
    }
    const int W = T.W;
    const int P = W | 1;
    const int TRc = TR + (bound ? 1 : 0);         // (the bound of row r0+TR-1 also needs row r0+TR)
    const int CP = (TRc * P) | 1;                 // odd tile pitch per column: conflict-free both ways
    double* tile = reinterpret_cast<double*>(tsm);             // [32][CP]
    double* lw_s = tile + 32 * CP;                             // [NW][32][W]
    int* cw_s = reinterpret_cast<int*>(lw_s + NW * 32 * W);    // [32][W]
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * TR;
    const int rows = G.order[0], stride0 = G.stride[0];
    for (int k = threadIdx.x; k < 32 * W; k += blockDim.x) {
        const int lc = k / W, w = k - lc * W;
        const int c = min(c0 + lc, T.n_cols - 1);
        const int64_t f = ((int64_t)c * T.tiles_per_col * W + w) * 32;     // lane 0 of the column's first tile
        cw_s[k] = __ldg(T.cell_w + f);
#pragma unroll
        for (int j = 0; j < NW; ++j) lw_s[(j * 32 + lc) * W + w] = __ldg(T.lam_w + (int64_t)j * T.lam_w_plane + f);
    }
    __syncthreads();
    // (independent iterations: unrolled so that the gathers of several elements are in flight)
#pragma unroll 6
    for (int k = threadIdx.x; k < TRc * W * 32; k += blockDim.x) {
        const int lc = k & 31;
        const int rw = k >> 5;
        const int lr = rw / W, w = rw - lr * W;
        const int r = min(r0 + lr, rows - 1);
        double lam[D];
        lam[0] = 0.0;
#pragma unroll
        for (int j = 0; j < NW; ++j) lam[j + 1] = lw_s[(j * 32 + lc) * W + w];
        tile[lc * CP + lr * P + w] = Lerp<double, D, 1>::eval(Jprev, r * stride0 + cw_s[lc * W + w], G.stride, lam);
    }
    __syncthreads();
    const int nr = min(TR, rows - r0);
    for (int lc = threadIdx.x >> 5; lc < 32; lc += blockDim.x >> 5) {
        if (c0 + lc >= T.n_cols) break;
        if (T.col_pairs) {
            // two rows per lane: row q at q*P + (q >> 1) (see k_sweep_fact_column2)
            double* dstc = T.col_table + (int64_t)(c0 + lc) * pitch;
            for (int k = threadIdx.x & 31; k < nr * P; k += 32) {
                const int lr = k / P, w = k - lr * P, r = r0 + lr;
                dstc[r * P + (r >> 1) + w] = tile[lc * CP + k];
            }
        } else {
            double* dst = T.col_table + (int64_t)(c0 + lc) * pitch + (int64_t)r0 * P;
            for (int k = threadIdx.x & 31; k < nr * P; k += 32) dst[k] = tile[lc * CP + k];
        }
    }
    if (bound) {
        // (threads along the rows of a column: the 16-byte stores of a warp are contiguous)
        double2* dstb = reinterpret_cast<double2*>(T.col_bound);
        for (int k = threadIdx.x; k < 32 * nr; k += blockDim.x) {
            const int lc = k / nr, lr = k - lc * nr, q = r0 + lr;
            if (c0 + lc >= T.n_cols) break;
            dstb[(int64_t)(c0 + lc) * rows + q] =
                q < rows - 1 ? column_bound(tile + lc * CP + lr * P, P, W, PV) : make_double2(0.0, CUDART_NAN);
        }
    }
}

// probabilities of the column kernels as launch constants (1 for a deterministic system)
static PVals column_pvals(const SdpTables& T) {
    PVals pv;
    for (int w = 0; w < SDP_FACTORED_MAX_W_REG; ++w)
        pv.v[w] = (w < T.W) ? (T.expect ? T.p_host[w] : 1.0) : 0.0;
    return pv;
}
// whether the pre-pass writes SdpTables.col_bound (and the sweep may prune): depends on the
// tables and the grid only, so that a separate pre-pass (sdp_column_table) and the sweep agree
static bool column_bound_on(const GridT<double>& G, const SdpTables& T) {
    if (!T.col_bound || ((uintptr_t)T.col_bound & 15) || T.col_pairs || !(T.expect || T.W == 1))
        return false;
    if (SDP_COLUMN_PITCH(G.order[0], T.W) * 8 + (int64_t)G.order[0] * 16 > SDP_COLUMN_MAX_SMEM_BYTES) return false;
    const PVals pv = column_pvals(T);
    for (int w = 0; w < T.W; ++w)
        if (!(pv.v[w] >= 0.0 && pv.v[w] <= 1.0)) return false;
    return true;
}

template <int D>
static int launch_column_table(const GridT<double>& G, const SdpTables& T, const double* Jprev, cudaStream_t st) {
    constexpr int NW = D - 1;
    const int P = T.W | 1;
    // rows per CTA: 16, fewer when the shard has so few columns that 16 would leave SMs idle
    // (the 62 columns of one rank of eight: 250 CTAs of 16 rows, 1 000 of 4)
    int TR = SDP_CT_ROWS;
    const int64_t col_blocks = (T.n_cols + 31) / 32;
    while (TR > 4 && col_blocks * ((G.order[0] + TR - 1) / TR) < 148 * 6) TR >>= 1;
    const int bound = column_bound_on(G, T);
    const PVals pv = column_pvals(T);
    const size_t tshm = (size_t)32 * (((TR + bound) * P) | 1) * 8 + (size_t)NW * 32 * T.W * 8 + (size_t)32 * T.W * 4;
    dim3 grid((unsigned)col_blocks, (unsigned)((G.order[0] + TR - 1) / TR));
    const int64_t pitch = T.col_pairs ? SDP_COLUMN_PITCH2(G.order[0], T.W) : SDP_COLUMN_PITCH(G.order[0], T.W);
    if (g_wait_peers) {
        // the flag wait of the previous exchange rides in this kernel (sdp_sweep_partials_after)
        const PeersDev P2 = *g_wait_peers;
        g_wait_peers = nullptr;
        launch_pdl(k_column_table<D, true>, grid, dim3(256), tshm, st,
                   G, T, Jprev, pitch, P2, (unsigned long long)tuning().p2p_timeout_s * 1000000000ULL, TR, pv, bound);
    } else {
        PeersDev none;
        memset(&none, 0, sizeof(none));
        launch_pdl(k_column_table<D, false>, grid, dim3(256), tshm, st, G, T, Jprev, pitch, none, 0ULL, TR, pv, bound);
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// MAXT: launch bound (512 threads leave 128 registers per thread, 640 leave 102, 768 leave 85).
// prepass: 0 = the CTA gathers its table from J_prev, 1 = copies it from col_table with
// vector loads, 2 = with one bulk asynchronous copy (TMA engine, SASS UBLKCP) on an mbarrier.
// PRUNE: the column's bound (SdpTables.col_bound) comes with its table, behind it in shared
// memory; a group of UB controls is skipped when no lane needs any of them (column_skip: it
// provably loses against the lane's best so far).  Each lane first evaluates the control it
// chose in the previous sweep (part_idx, when it is a control of the item), so that the best
// is good from the first group on.  The minimum over the controls, ties to the lowest index
// (`better`), does not depend on the order they are visited in: the results are those of
// PRUNE = false, bit for bit.  `stats` (optional): warp steps met and skipped.
template <int D, int WM, int UB, int PF, bool FULL, int MAXT, bool PRUNE>     // FULL: W == WM, every slot live
__global__ void __launch_bounds__(MAXT, 1)
k_sweep_fact_column(GridT<double> G, SdpTables T, const double* __restrict__ Jprev,
                    double* __restrict__ part_val, int32_t* __restrict__ part_idx,
                    double inv_stride0, PVals PV, int64_t pitch, int prepass, int dynamic,
                    double sum_p, unsigned long long* __restrict__ stats) {
    constexpr int NW = D - 1;
    extern __shared__ __align__(128) unsigned char csm[];
    __shared__ int next_item[2];                        // dynamic hand-out of the items of a column (two, used in turn)
    double* R_sh = reinterpret_cast<double*>(csm);      // [order[0]][P] + slack = `pitch` doubles
    const double2* B_sh = reinterpret_cast<const double2*>(csm + pitch * 8);     // PRUNE: [order[0]] (m, A)
    __shared__ int cw_sh[WM];
    __shared__ double lw_sh[NW][WM];
    __shared__ __align__(8) uint64_t tbar;              // completion of the bulk copy of a table
    uint32_t tphase = 0;
    if (threadIdx.x == 0) {
        mbar_init(smem_u32(&tbar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        next_item[0] = next_item[1] = 0;
    }
    cudaGridDependencySynchronize();       // (programmatic dependent launch: the pre-pass's column tables)
    __syncthreads();
    const int W = T.W;
    const int P = W | 1;        // odd row pitch: adjacent rows never share a bank pair
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int rows = G.order[0];
    const int stride0 = G.stride[0];

    int64_t i = T.seg_begin[blockIdx.x];
    const int64_t seg_end = T.seg_begin[blockIdx.x + 1];
    int turn = 0;                    // which of the two item counters this column run uses
    while (i < seg_end) {
        // (positions i index the item list directly, or through T.item_order: the bands of a
        // column back to back, so that a device-resident sweep loads each column's table once)
        const int col = T.items[T.item_order ? T.item_order[i] : i].Upad;     // the column of the item's tile
        const int64_t run_end = T.run_end[i];     // end of the run of positions sharing this table
        const int64_t e = run_end < seg_end ? run_end : seg_end;
        __syncthreads();                 // the previous column's readers are done with R
        // (the counter of the NEXT run is cleared now: nobody touches it during this run)
        if (threadIdx.x == 0) next_item[turn ^ 1] = 0;
        // prepass 2: the table arrives by bulk copy while the warps already take their first item
        // and issue its first loads from the (x,u) stream; each thread waits on the copy's barrier
        // just before its first read of the table (`have_table`)
        bool have_table = prepass < 2;
        if (prepass >= 2) {
            // the column's table, tabulated by k_column_table, is one contiguous block: one
            // thread hands it to the TMA engine in <= 32 KB pieces
            if (threadIdx.x == 0) {
                const unsigned char* src = reinterpret_cast<const unsigned char*>(T.col_table + (int64_t)col * pitch);
                const uint32_t bytes = (uint32_t)(pitch * 8);
                const uint32_t bbytes = PRUNE ? (uint32_t)rows * 16u : 0u;
                const uint32_t bar = smem_u32(&tbar);
                mbar_expect_tx(bar, bytes + bbytes);
                for (uint32_t o = 0; o < bytes; o += 32768u)
                    bulk_g2s(smem_u32(csm + o), src + o, min(32768u, bytes - o), bar);
                if (PRUNE) {
                    // the bound, on the same barrier
                    const unsigned char* bsrc = reinterpret_cast<const unsigned char*>(T.col_bound + (int64_t)col * rows * 2);
                    for (uint32_t o = 0; o < bbytes; o += 32768u)
                        bulk_g2s(smem_u32(csm + bytes + o), bsrc + o, min(32768u, bbytes - o), bar);
                }
            }
            if (prepass == 2) {          // (3: the wait moves behind the first item's loads)
                mbar_wait(smem_u32(&tbar), tphase);
                have_table = true;
            }
        } else if (prepass) {
            const double2* __restrict__ src = reinterpret_cast<const double2*>(T.col_table + (int64_t)col * pitch);
            double2* dst = reinterpret_cast<double2*>(R_sh);
            const int n2 = (int)(pitch >> 1);
            int k = threadIdx.x;
            for (; k + 7 * (int)blockDim.x < n2; k += 8 * blockDim.x) {     // 8 independent loads in flight
                double2 v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = src[k + j * blockDim.x];
#pragma unroll
                for (int j = 0; j < 8; ++j) dst[k + j * blockDim.x] = v[j];
            }
            for (; k < n2; k += blockDim.x) dst[k] = src[k];
            if (PRUNE) {
                const double2* __restrict__ bsrc = reinterpret_cast<const double2*>(T.col_bound + (int64_t)col * rows * 2);
                double2* bdst = reinterpret_cast<double2*>(R_sh + pitch);
                for (int r = threadIdx.x; r < rows; r += blockDim.x) bdst[r] = bsrc[r];
            }
        } else {
            if (threadIdx.x < W) {
                // the column's w-part: lane 0 of its first tile
                const int64_t f = ((int64_t)col * T.tiles_per_col * W + threadIdx.x) * 32;
                cw_sh[threadIdx.x] = __ldg(T.cell_w + f);
#pragma unroll
                for (int k = 0; k < NW; ++k)
                    lw_sh[k][threadIdx.x] = __ldg(T.lam_w + (int64_t)k * T.lam_w_plane + f);
            }
            __syncthreads();
            for (int idx = threadIdx.x; idx < rows * W; idx += blockDim.x) {
                const int r = idx / W, w = idx - r * W;
                double lam[D];
                lam[0] = 0.0;
#pragma unroll
                for (int k = 0; k < NW; ++k) lam[k + 1] = lw_sh[k][w];
                R_sh[r * P + w] = Lerp<double, D, 1>::eval(Jprev, r * stride0 + cw_sh[w], G.stride, lam);
            }
            if (PRUNE) {
                __syncthreads();
                double2* bdst = reinterpret_cast<double2*>(R_sh + pitch);
                for (int r = threadIdx.x; r < rows; r += blockDim.x)
                    bdst[r] = r < rows - 1 ? column_bound(R_sh + r * P, P, W, PV) : make_double2(0.0, CUDART_NAN);
            }
        }
        if (prepass < 2) __syncthreads();

        // the warps share the items of the column: round-robin, or (dynamic) first come first
        // served - the items differ in length and a column piece may hold only a few of them
        for (int round = 0;; ++round) {
            int k = round * nwarps + warp;
            if (dynamic) {
                if (lane == 0) k = atomicAdd(&next_item[turn], 1);
                k = __shfl_sync(0xffffffffu, k, 0);
            }
            const int64_t pos = i + k;
            if (pos >= e) break;
            const int64_t item_id = T.item_order ? T.item_order[pos] : pos;
            const SdpItem it = T.items[item_id];
            const int Us = T.U[(int64_t)it.state * 32 + lane];      // by position; 0 on padding lanes
            const int32_t* __restrict__ cup = T.cell + it.entry_base + lane;
            const double* __restrict__ lup = T.lam + it.entry_base + lane;
            const double* __restrict__ gp = T.g + it.g_base + lane;
            double best_v = CUDART_INF;
            int best_i = INT_MAX;
            const int last = it.u_count - 1;
            // PRUNE: the lane's choice of the previous sweep, if it is one of this item's controls
            // (read before this warp overwrites it below; any other value is ignored)
            int seed = -1;
            int c_s = 0;
            double g_s = 0.0, l_s = 0.0;
            if (PRUNE) {
                const int s = part_idx[item_id * 32 + lane];
                if (s >= it.u_begin && s - it.u_begin < it.u_count && s < Us) {
                    seed = s;
                    const int64_t o = (int64_t)(s - it.u_begin) * 32;
                    c_s = cup[o];
                    g_s = gp[o];
                    l_s = lup[o];
                }
            }
            int n_steps = 0, n_skipped = 0;

            // PF groups of UB controls are in flight: group k of the run sits in stage k % PF
            // (rows past the run repeat its last row)
            int c_n[PF][UB];
            double g_n[PF][UB], l_n[PF][UB];
#pragma unroll
            for (int s = 0; s < PF; ++s)
#pragma unroll
                for (int b = 0; b < UB; ++b) {
                    const int64_t o = (int64_t)min(s * UB + b, last) * 32;
                    c_n[s][b] = __ldcs(cup + o);
                    g_n[s][b] = __ldcs(gp + o);
                    l_n[s][b] = __ldcs(lup + o);
                }
            if (!have_table) {           // (warp-uniform; first item of the run only)
                mbar_wait(smem_u32(&tbar), tphase);
                have_table = true;
            }
            if (PRUNE && seed >= 0) {
                // the seed, evaluated with the very operations of the loop below
                const double oml = sub_(1.0, l_s);
                const int q = __double2int_rn(__dmul_rn((double)c_s, inv_stride0));
                const double* Ra = R_sh + q * P;
                double acc = 0.0;
#pragma unroll
                for (int w = 0; w < WM; ++w) {
                    const double v = add_(mul_(oml, Ra[w]), mul_(l_s, Ra[P + w]));
                    const double jg = add_(g_s, v);
                    const double nxt = T.expect ? add_(acc, mul_(jg, PV.v[w])) : jg;
                    acc = (FULL || w < W) ? nxt : acc;
                }
                if (better(acc, seed, best_v, best_i)) {
                    best_v = acc;
                    best_i = seed;
                }
            }
            for (int uu0 = 0; uu0 < it.u_count; uu0 += UB * PF) {
#pragma unroll
                for (int s = 0; s < PF; ++s) {
                    const int uu = uu0 + s * UB;
                    if (uu < it.u_count) {                    // warp-uniform
                        double gv[UB], lu[UB], oml[UB];
                        const double* Ra[UB];
                        bool need = !PRUNE;
#pragma unroll
                        for (int b = 0; b < UB; ++b) {
                            gv[b] = g_n[s][b];
                            lu[b] = l_n[s][b];
                            oml[b] = sub_(1.0, lu[b]);
                            // row q0 = cell_u / stride0 exactly (cell_u is a multiple of stride0
                            // below 2^31; padding entries hold cell 0)
                            const int q = __double2int_rn(__dmul_rn((double)c_n[s][b], inv_stride0));
                            Ra[b] = R_sh + q * P;
                            // (padding lanes and rows past the run never need a control)
                            if (PRUNE && uu + b <= last && it.u_begin + uu + b < Us)
                                need |= !column_skip(B_sh[q], gv[b], lu[b], sum_p, best_v);
                        }
                        if (uu + UB * PF < it.u_count) {
#pragma unroll
                            for (int b = 0; b < UB; ++b) {
                                const int64_t o = (int64_t)min(uu + UB * PF + b, last) * 32;
                                c_n[s][b] = __ldcs(cup + o);
                                g_n[s][b] = __ldcs(gp + o);
                                l_n[s][b] = __ldcs(lup + o);
                            }
                        }
                        if (PRUNE) {
                            ++n_steps;
                            if (!__any_sync(0xffffffffu, need)) {
                                ++n_skipped;
                                continue;
                            }
                        }
                        // slots >= W read past the W live values of a row (its pad, the next row,
                        // or the slack behind the table) and are discarded below: no guards
                        double v[UB][WM];
#pragma unroll
                        for (int b = 0; b < UB; ++b)
#pragma unroll
                            for (int w = 0; w < WM; ++w)
                                v[b][w] = add_(mul_(oml[b], Ra[b][w]), mul_(lu[b], Ra[b][P + w]));
#pragma unroll
                        for (int b = 0; b < UB; ++b) {
                            double acc = 0.0;
#pragma unroll
                            for (int w = 0; w < WM; ++w) {
                                const double jg = add_(gv[b], v[b][w]);
                                const double nxt = T.expect ? add_(acc, mul_(jg, PV.v[w])) : jg;
                                acc = (FULL || w < W) ? nxt : acc;   // slots past W do not take part
                            }
                            const int u = it.u_begin + uu + b;
                            if (uu + b <= last && u < Us && better(acc, u, best_v, best_i)) {
                                best_v = acc;
                                best_i = u;
                            }
                        }
                    }
                }
            }
            part_val[item_id * 32 + lane] = best_v;
            part_idx[item_id * 32 + lane] = best_i;
            if (PRUNE && stats && lane == 0) {
                atomicAdd(stats, (unsigned long long)n_steps);
                atomicAdd(stats + 1, (unsigned long long)n_skipped);
            }
        }
        if (prepass >= 2) {
            // a warp that got no item of this run still observes the copy's completion: thread 0
            // re-arms the barrier for the next table only after every thread has seen this phase
            if (!have_table) mbar_wait(smem_u32(&tbar), tphase);
            tphase ^= 1u;
        }
        turn ^= 1;
        i = e;
    }
}

// pruning sweep: warp steps met / skipped, counted with "col_prune_stats" (sdp_col_prune_counts)
static unsigned long long* g_prune_stats = nullptr;
extern "C" int sdp_col_prune_counts(int64_t* steps, int64_t* skipped) {
    if (!steps || !skipped) return fail(SDP_EINVAL, "%s", "sdp_col_prune_counts: NULL pointer");
    *steps = *skipped = 0;
    if (!g_prune_stats) return SDP_OK;
    unsigned long long h[2];
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(h, g_prune_stats, sizeof(h), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemset(g_prune_stats, 0, sizeof(h));
    if (e != cudaSuccess) return fail(SDP_ECUDA, "sdp_col_prune_counts: %s", cudaGetErrorString(e));
    *steps = (int64_t)h[0];
    *skipped = (int64_t)h[1];
    return SDP_OK;
}

template <int D, int WM, int UB, int PF, int MAXT, bool PRUNE>
static int set_column_attrs(size_t shm) {
    static size_t attr_set = 0;          // per instantiation
    if (attr_set >= shm) return SDP_OK;
    cudaError_t e = cudaFuncSetAttribute(k_sweep_fact_column<D, WM, UB, PF, true, MAXT, PRUNE>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(k_sweep_fact_column<D, WM, UB, PF, false, MAXT, PRUNE>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm);
    // the largest shared-memory carve-out (the kernel streams with evict-first loads: 2 % L1 hit
    // rate): k_combine_column_small asks for the same one, so that one of its CTAs can join a
    // resident CTA of this kernel without the SM draining to change its configuration
    if (e == cudaSuccess && tuning().carveout)
        e = cudaFuncSetAttribute(k_sweep_fact_column<D, WM, UB, PF, true, MAXT, PRUNE>,
                                 cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e == cudaSuccess && tuning().carveout)
        e = cudaFuncSetAttribute(k_sweep_fact_column<D, WM, UB, PF, false, MAXT, PRUNE>,
                                 cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return fail(SDP_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = shm;
    return SDP_OK;
}

template <int D, int WM, int UB, int PF, int MAXT, bool PRUNE>
static void launch_fact_column_kp(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                                  double* part_val, int32_t* part_idx, cudaStream_t st, int threads, size_t shm,
                                  int64_t pitch, int prepass, double sum_p, unsigned long long* stats) {
    const PVals pv = column_pvals(T);
    const double inv0 = 1.0 / (double)G.stride[0];
    const int dynamic = (T.col_launch_hint & 0xffff) ? !((T.col_launch_hint >> 16) & 1) : tuning().col_dynamic;
    if (T.W == WM)
        launch_pdl(k_sweep_fact_column<D, WM, UB, PF, true, MAXT, PRUNE>, dim3((unsigned)T.n_segs), dim3(threads),
                   shm, st, G, T, Jprev, part_val, part_idx, inv0, pv, pitch, prepass, dynamic, sum_p, stats);
    else
        launch_pdl(k_sweep_fact_column<D, WM, UB, PF, false, MAXT, PRUNE>, dim3((unsigned)T.n_segs), dim3(threads),
                   shm, st, G, T, Jprev, part_val, part_idx, inv0, pv, pitch, prepass, dynamic, sum_p, stats);
}

template <int D, int WM, int UB, int PF, int MAXT>
static int launch_fact_column_k(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                                double* part_val, int32_t* part_idx, cudaStream_t st, int threads) {
    const int64_t pitch = SDP_COLUMN_PITCH(G.order[0], T.W);
    if ((size_t)pitch * 8 > SDP_COLUMN_MAX_SMEM_BYTES)
        return fail(SDP_EINVAL, "%s", "sdp_sweep: layout CF: the column table does not fit shared memory");
    const int prepass = tuning().col_prepass;
    if (prepass && !T.col_table_ready) {
        int rc = launch_column_table<D>(G, T, Jprev, st);
        if (rc) return rc;
    }
    const bool prune = tuning().col_prune && column_bound_on(G, T);
    const size_t shm = (size_t)pitch * 8 + (prune ? (size_t)G.order[0] * 16 : 0);
    int rc = prune ? set_column_attrs<D, WM, UB, PF, MAXT, true>(shm) : set_column_attrs<D, WM, UB, PF, MAXT, false>(shm);
    if (rc) return rc;
    if (prune) {
        unsigned long long* stats = nullptr;
        if (tuning().col_prune_stats) {
            if (!g_prune_stats) {
                cudaError_t e = cudaMalloc(&g_prune_stats, 2 * sizeof(unsigned long long));
                if (e == cudaSuccess) e = cudaMemset(g_prune_stats, 0, 2 * sizeof(unsigned long long));
                if (e != cudaSuccess) {
                    g_prune_stats = nullptr;
                    return fail(SDP_ECUDA, "col_prune_stats: %s", cudaGetErrorString(e));
                }
            }
            stats = g_prune_stats;
        }
        const PVals pv = column_pvals(T);
        double sum_p = 0.0;                  // (in w order: tablebuild.column_prune_skip)
        for (int w = 0; w < T.W; ++w) sum_p += pv.v[w];
        launch_fact_column_kp<D, WM, UB, PF, MAXT, true>(G, T, Jprev, part_val, part_idx, st, threads, shm, pitch,
                                                         prepass, sum_p, stats);
    } else {
        launch_fact_column_kp<D, WM, UB, PF, MAXT, false>(G, T, Jprev, part_val, part_idx, st, threads, shm, pitch,
                                                          prepass, 0.0, nullptr);
    }
    note_kernel("%sk_sweep_fact_column<%d,%d,%d,%d,%s,%d%s> [%d CTAs x %d threads]",
                (prepass && !T.col_table_ready) ? "k_column_table + " : "", D, WM, UB, PF,
                T.W == WM ? "true" : "false", MAXT, prune ? ",prune" : "", (int)T.n_segs, threads);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// Layout CF, two rows per lane (SdpTables.col_pairs).  ncu on k_sweep_fact_column: shared-memory
// wavefronts at 88 % of the pipe - 16 bytes of table per backup, R[q][w] and R[q+1][w] - with the
// fp64 pipe at 61 %.  Two rows of a column that are neighbours on axis 0 and have the same
// control grid land, for the same control, in the same or in neighbouring table rows
// (E' = E + P*dt: q' - q in {0, 1}), so a lane that owns both reads R[q], R[q+1], R[q'+1]: 3
// reads for 2 backups, 12 bytes per backup.  Lane l of a warp owns the positions 2j, 2j+1
// (j = l & 15) of the first (l < 16) or the second tile of a PAIR of tiles of the column; the
// u-part streams as int2 / double2.  Any other q' - q costs the warp a 4th read for that control.
// The table is swizzled, row q at q*P + (q >> 1): a lane step of two rows is then an odd number
// of doubles (2P + 1) and a half-warp's 8-byte reads still cover all 32 banks.
// Same operations per backup, in the same order, as every other layout: bit-identical.
// ---------------------------------------------------------------------------
template <int D, int WM, bool FULL, int MAXT>
__global__ void __launch_bounds__(MAXT, 1)
k_sweep_fact_column2(GridT<double> G, SdpTables T, double* __restrict__ part_val,
                     int32_t* __restrict__ part_idx, double inv_stride0, PVals PV, int64_t pitch, int dynamic) {
    extern __shared__ __align__(128) unsigned char csm[];
    __shared__ int next_item;
    __shared__ __align__(8) uint64_t tbar;
    double* R_sh = reinterpret_cast<double*>(csm);
    uint32_t tphase = 0;
    if (threadIdx.x == 0) {
        mbar_init(smem_u32(&tbar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int W = T.W;
    const int P = W | 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int half = lane >> 4, j2 = (lane & 15) * 2;

    int64_t i = T.seg_begin[blockIdx.x];
    const int64_t seg_end = T.seg_begin[blockIdx.x + 1];
    while (i < seg_end) {
        const int col = T.items[T.item_order[i]].Upad;
        const int64_t run_end = T.run_end[i];
        const int64_t e = run_end < seg_end ? run_end : seg_end;
        __syncthreads();                 // the previous column's readers are done with R
        if (threadIdx.x == 0) {
            next_item = 0;
            const unsigned char* src = reinterpret_cast<const unsigned char*>(T.col_table + (int64_t)col * pitch);
            const uint32_t bytes = (uint32_t)(pitch * 8);
            const uint32_t bar = smem_u32(&tbar);
            mbar_expect_tx(bar, bytes);
            for (uint32_t o = 0; o < bytes; o += 32768u)
                bulk_g2s(smem_u32(csm + o), src + o, min(32768u, bytes - o), bar);
        }
        mbar_wait(smem_u32(&tbar), tphase);
        tphase ^= 1u;
        __syncthreads();

        for (int round = 0;; ++round) {
            int k = round * nwarps + warp;
            if (dynamic) {
                if (lane == 0) k = atomicAdd(&next_item, 1);
                k = __shfl_sync(0xffffffffu, k, 0);
            }
            const int64_t pos = i + k;
            if (pos >= e) break;
            const int64_t idA = T.item_order[pos];
            const SdpItem itA = T.items[idA];
            const int64_t idB = itA.g_base;           // the same run of controls in the pair's second tile
            const bool live = !half || idB >= 0;
            const int64_t my_id = (half && idB >= 0) ? idB : idA;
            int64_t ebase = itA.entry_base;
            int tile = itA.state;
            if (half && idB >= 0) {
                ebase = T.items[idB].entry_base;
                tile = T.items[idB].state;
            }
            int Us0 = 0, Us1 = 0;
            if (live) {
                const int2 uu = *reinterpret_cast<const int2*>(T.U + (int64_t)tile * 32 + j2);
                Us0 = uu.x;
                Us1 = uu.y;
            }
            // control u of the tile: entries ebase + u*32 + position
            const int2* __restrict__ cup = reinterpret_cast<const int2*>(T.cell + ebase + j2);
            const double2* __restrict__ lup = reinterpret_cast<const double2*>(T.lam + ebase + j2);
            const double2* __restrict__ gp = reinterpret_cast<const double2*>(T.g + ebase + j2);
            const int cnt = itA.u_count, last = cnt - 1;
            double bv0 = CUDART_INF, bv1 = CUDART_INF;
            int bi0 = INT_MAX, bi1 = INT_MAX;

            int2 c_n[2];
            double2 l_n[2], g_n[2];
#pragma unroll
            for (int s2 = 0; s2 < 2; ++s2) {
                const int o = min(s2, last) * 16;
                c_n[s2] = __ldcs(cup + o);
                l_n[s2] = __ldcs(lup + o);
                g_n[s2] = __ldcs(gp + o);
            }
            for (int uu0 = 0; uu0 < cnt; uu0 += 2) {
#pragma unroll
                for (int s2 = 0; s2 < 2; ++s2) {
                    const int uu = uu0 + s2;
                    if (uu < cnt) {                         // warp-uniform
                        const int2 c = c_n[s2];
                        const double2 l = l_n[s2], g = g_n[s2];
                        if (uu + 2 < cnt) {
                            const int o = min(uu + 2, last) * 16;
                            c_n[s2] = __ldcs(cup + o);
                            l_n[s2] = __ldcs(lup + o);
                            g_n[s2] = __ldcs(gp + o);
                        }
                        const int qa = __double2int_rn(__dmul_rn((double)c.x, inv_stride0));
                        const int qb = __double2int_rn(__dmul_rn((double)c.y, inv_stride0));
                        const int dq = qb - qa;
                        const double* __restrict__ Ra0 = R_sh + qa * P + (qa >> 1);
                        const double* __restrict__ Ra1 = R_sh + (qa + 1) * P + ((qa + 1) >> 1);
                        const double* __restrict__ Rb1 = R_sh + (qb + 1) * P + ((qb + 1) >> 1);
                        const double oma = sub_(1.0, l.x), omb = sub_(1.0, l.y);
                        double acc0 = 0.0, acc1 = 0.0;
                        if (__any_sync(0xffffffffu, (unsigned)dq > 1u)) {
                            // rows that are no neighbours in the table: four reads
                            const double* __restrict__ Rb0 = R_sh + qb * P + (qb >> 1);
#pragma unroll
                            for (int w = 0; w < WM; ++w) {
                                const double va = add_(mul_(oma, Ra0[w]), mul_(l.x, Ra1[w]));
                                const double vb = add_(mul_(omb, Rb0[w]), mul_(l.y, Rb1[w]));
                                const double ja = add_(g.x, va), jb = add_(g.y, vb);
                                const double na = T.expect ? add_(acc0, mul_(ja, PV.v[w])) : ja;
                                const double nb = T.expect ? add_(acc1, mul_(jb, PV.v[w])) : jb;
                                acc0 = (FULL || w < W) ? na : acc0;
                                acc1 = (FULL || w < W) ? nb : acc1;
                            }
                        } else {
#pragma unroll
                            for (int w = 0; w < WM; ++w) {
                                const double x0 = Ra0[w], x1 = Ra1[w], x2 = Rb1[w];
                                const double y0 = dq ? x1 : x0;           // R[qb][w]
                                const double va = add_(mul_(oma, x0), mul_(l.x, x1));
                                const double vb = add_(mul_(omb, y0), mul_(l.y, x2));
                                const double ja = add_(g.x, va), jb = add_(g.y, vb);
                                const double na = T.expect ? add_(acc0, mul_(ja, PV.v[w])) : ja;
                                const double nb = T.expect ? add_(acc1, mul_(jb, PV.v[w])) : jb;
                                acc0 = (FULL || w < W) ? na : acc0;
                                acc1 = (FULL || w < W) ? nb : acc1;
                            }
                        }
                        const int u = itA.u_begin + uu;
                        if (u < Us0 && better(acc0, u, bv0, bi0)) { bv0 = acc0; bi0 = u; }
                        if (u < Us1 && better(acc1, u, bv1, bi1)) { bv1 = acc1; bi1 = u; }
                    }
                }
            }
            if (live) {
                *reinterpret_cast<double2*>(part_val + my_id * 32 + j2) = make_double2(bv0, bv1);
                *reinterpret_cast<int2*>(part_idx + my_id * 32 + j2) = make_int2(bi0, bi1);
            }
        }
        i = e;
    }
}

template <int D, int WM, int MAXT>
static int launch_fact_column2_k(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                                 double* part_val, int32_t* part_idx, cudaStream_t st, int threads) {
    const int64_t pitch = SDP_COLUMN_PITCH2(G.order[0], T.W);
    const size_t shm = (size_t)pitch * 8;
    if (shm > SDP_COLUMN_MAX_SMEM_BYTES)
        return fail(SDP_EINVAL, "%s", "sdp_sweep: layout CF: the column table does not fit shared memory");
    if (!T.item_order || !T.pos_row)
        return fail(SDP_EINVAL, "%s", "sdp_sweep: layout CF with col_pairs needs item_order and pos_row");
    if (!T.col_table_ready) {
        int rc = launch_column_table<D>(G, T, Jprev, st);
        if (rc) return rc;
    }
    static size_t attr_set = 0;          // per instantiation
    if (attr_set < shm) {
        cudaError_t e = cudaFuncSetAttribute(k_sweep_fact_column2<D, WM, true, MAXT>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(k_sweep_fact_column2<D, WM, false, MAXT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm);
        if (e != cudaSuccess) return fail(SDP_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        attr_set = shm;
    }
    PVals pv;
    for (int w = 0; w < SDP_FACTORED_MAX_W_REG; ++w)
        pv.v[w] = (w < T.W) ? (T.expect ? T.p_host[w] : 1.0) : 0.0;
    const double inv0 = 1.0 / (double)G.stride[0];
    const int dynamic = (T.col_launch_hint & 0xffff) ? !((T.col_launch_hint >> 16) & 1) : tuning().col_dynamic;
    if (T.W == WM)
        k_sweep_fact_column2<D, WM, true, MAXT><<<(unsigned)T.n_segs, threads, shm, st>>>(
            G, T, part_val, part_idx, inv0, pv, pitch, dynamic);
    else
        k_sweep_fact_column2<D, WM, false, MAXT><<<(unsigned)T.n_segs, threads, shm, st>>>(
            G, T, part_val, part_idx, inv0, pv, pitch, dynamic);
    note_kernel("%sk_sweep_fact_column2<%d,%d,%s,%d> [%d CTAs x %d threads]",
                !T.col_table_ready ? "k_column_table + " : "", D, WM, T.W == WM ? "true" : "false", MAXT,
                (int)T.n_segs, threads);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

template <int D, int WM>
static int launch_fact_column2_w(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                                 double* part_val, int32_t* part_idx, cudaStream_t st) {
    const int hint_threads = T.col_launch_hint & 0xffff;
    const int threads = hint_threads ? clampi(hint_threads, 128, 768) / 32 * 32 : (tuning().col_threads ? tuning().col_threads : 768);
    if (threads > 640) return launch_fact_column2_k<D, WM, 768>(G, T, Jprev, part_val, part_idx, st, threads);
    return launch_fact_column2_k<D, WM, 640>(G, T, Jprev, part_val, part_idx, st, threads);
}

template <int D, int WM>
static int launch_fact_column_w(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                                double* part_val, int32_t* part_idx, cudaStream_t st) {
    // T.col_launch_hint (low 16 bits: threads per CTA, bit 16: hand the items out round-robin):
    // the caller's knowledge of the launch - many short column pieces per CTA (a band of rows)
    // run best with 640 threads round-robin, long ones with 768 and first come first served
    const int hint_threads = T.col_launch_hint & 0xffff;
    const int ub = tuning().col_ub, pf = tuning().col_pf;
    // default CTA size: 768 threads (one group of 2 controls in flight per lane); the pruning sweep
    // skips ~94 % of the evaluations of config #5 and is then bound by the latency of the (x,u)
    // stream, which 640 threads with two groups in flight hide better: 1.003 against 1.044 ms per
    // sweep (profiles/r3_prune_timing.json, "launch_shapes")
    const int auto_threads = (tuning().col_prune && column_bound_on(G, T)) ? 640 : 768;
    const int threads = hint_threads ? clampi(hint_threads, 128, 768) / 32 * 32
                                     : (tuning().col_threads ? tuning().col_threads : auto_threads);
    if (threads > 640) {       // 85 registers per thread
        if (ub == 2) return launch_fact_column_k<D, WM, 2, 1, 768>(G, T, Jprev, part_val, part_idx, st, threads);
        return pf == 2 ? launch_fact_column_k<D, WM, 1, 2, 768>(G, T, Jprev, part_val, part_idx, st, threads)
                       : launch_fact_column_k<D, WM, 1, 1, 768>(G, T, Jprev, part_val, part_idx, st, threads);
    }
    if (threads > 512)
        return pf == 2 ? launch_fact_column_k<D, WM, 2, 2, 640>(G, T, Jprev, part_val, part_idx, st, threads)
                       : launch_fact_column_k<D, WM, 2, 1, 640>(G, T, Jprev, part_val, part_idx, st, threads);
    if (ub == 2)
        return pf == 2 ? launch_fact_column_k<D, WM, 2, 2, 512>(G, T, Jprev, part_val, part_idx, st, threads)
                       : launch_fact_column_k<D, WM, 2, 1, 512>(G, T, Jprev, part_val, part_idx, st, threads);
    return pf == 2 ? launch_fact_column_k<D, WM, 1, 2, 512>(G, T, Jprev, part_val, part_idx, st, threads)
                   : launch_fact_column_k<D, WM, 1, 1, 512>(G, T, Jprev, part_val, part_idx, st, threads);
}

template <int D>
static int launch_fact_column(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                              double* part_val, int32_t* part_idx, cudaStream_t st) {
    if (T.col_pairs) {
        if (tuning().col_prepass < 2)
            return fail(SDP_EINVAL, "%s", "sdp_sweep: layout CF with col_pairs needs col_prepass >= 2");
        if (T.W <= 3) return launch_fact_column2_w<D, 3>(G, T, Jprev, part_val, part_idx, st);
        if (T.W <= 5) return launch_fact_column2_w<D, 5>(G, T, Jprev, part_val, part_idx, st);
        return launch_fact_column2_w<D, 9>(G, T, Jprev, part_val, part_idx, st);
    }
    if (T.W <= 3) return launch_fact_column_w<D, 3>(G, T, Jprev, part_val, part_idx, st);
    if (T.W <= 5) return launch_fact_column_w<D, 5>(G, T, Jprev, part_val, part_idx, st);
    return launch_fact_column_w<D, 9>(G, T, Jprev, part_val, part_idx, st);
}

template <int D, int MASK>
static int launch_fact_m(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                         double* part_val, int32_t* part_idx, cudaStream_t st) {
    if (T.layout == SDP_LAYOUT_STATE_MINOR_FACTORED) {
        // register slots for the w-part: the smallest of 3 / 5 / 9 that holds W
        if (T.W <= 3) launch_fact_tiled_w<D, MASK, 3>(G, T, Jprev, part_val, part_idx, st);
        else if (T.W <= 5) launch_fact_tiled_w<D, MASK, 5>(G, T, Jprev, part_val, part_idx, st);
        else launch_fact_tiled_w<D, MASK, SDP_FACTORED_MAX_W_REG>(G, T, Jprev, part_val, part_idx, st);
    } else {
        const int warps = 8;
        constexpr int NW = Fact<D, MASK>::NW;
        unsigned blocks = (unsigned)((T.n_items + warps - 1) / warps);
        if (MASK == 1 && tuning().hoist) {
            // rows of the per-item inner-interpolation table that fit 44 KB of shared memory
            const long budget = (44L * 1024 - 8L * T.W) / warps - (long)T.W * (8 * NW + 4);
            int RP = (int)(budget / (8L * T.W)) - 1;
            if (RP > 32) RP = 32;
            if (RP >= 2 && T.W <= SDP_FACTORED_MAX_W_REG && T.p_host && tuning().hoist_const) {
                // constant-W kernel: no p[] in shared memory (same row budget, slightly smaller block)
                size_t shm = (size_t)warps * ((size_t)T.W * (RP + 1 + NW) * 8 + (size_t)T.W * 4);
                const double inv0 = 1.0 / (double)G.stride[0];
                PVals pv;
                for (int w = 0; w < SDP_FACTORED_MAX_W_REG; ++w)
                    pv.v[w] = (w < T.W) ? (T.expect ? T.p_host[w] : 1.0) : 0.0;
                if (T.W <= 3)
                    k_sweep_fact_hoist_c<D, 3><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx, RP, inv0, pv);
                else if (T.W <= 5)
                    k_sweep_fact_hoist_c<D, 5><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx, RP, inv0, pv);
                else
                    k_sweep_fact_hoist_c<D, 9><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx, RP, inv0, pv);
                note_kernel("k_sweep_fact_hoist_c<%d,%d>", D, T.W <= 3 ? 3 : (T.W <= 5 ? 5 : 9));
                SDP_LAUNCH_CHECK();
                return SDP_OK;
            }
            if (RP >= 2) {
                size_t shm = (size_t)T.W * 8 + (size_t)warps * ((size_t)T.W * (RP + 1 + NW) * 8 + (size_t)T.W * 4);
                const double inv0 = 1.0 / (double)G.stride[0];   // host side: keeps fp64 division out of the kernel
                if (tuning().hoist_upl == 2)
                    k_sweep_fact_hoist<D, 2><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx, RP, inv0);
                else
                    k_sweep_fact_hoist<D, 4><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx, RP, inv0);
                note_kernel("k_sweep_fact_hoist<%d,%d>", D, tuning().hoist_upl == 2 ? 2 : 4);
                SDP_LAUNCH_CHECK();
                return SDP_OK;
            }
        }
        size_t shm = (size_t)T.W * 8 + (size_t)warps * T.W * (8 * NW + 4);
        if (tuning().upl == 2)
            k_sweep_fact<D, MASK, 2><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx);
        else
            k_sweep_fact<D, MASK, 4><<<blocks, warps * 32, shm, st>>>(G, T, Jprev, part_val, part_idx);
        note_kernel("k_sweep_fact<%d,%d,%d>", D, MASK, tuning().upl == 2 ? 2 : 4);
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

template <int D>
static int launch_fact(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                       double* part_val, int32_t* part_idx, cudaStream_t st);
template <>
int launch_fact<2>(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                   double* part_val, int32_t* part_idx, cudaStream_t st) {
    switch (T.u_mask) {
        case 1: return launch_fact_m<2, 1>(G, T, Jprev, part_val, part_idx, st);
        default: return launch_fact_m<2, 2>(G, T, Jprev, part_val, part_idx, st);
    }
}
template <>
int launch_fact<3>(const GridT<double>& G, const SdpTables& T, const double* Jprev,
                   double* part_val, int32_t* part_idx, cudaStream_t st) {
    switch (T.u_mask) {
        case 1: return launch_fact_m<3, 1>(G, T, Jprev, part_val, part_idx, st);
        case 2: return launch_fact_m<3, 2>(G, T, Jprev, part_val, part_idx, st);
        case 3: return launch_fact_m<3, 3>(G, T, Jprev, part_val, part_idx, st);
        case 4: return launch_fact_m<3, 4>(G, T, Jprev, part_val, part_idx, st);
        case 5: return launch_fact_m<3, 5>(G, T, Jprev, part_val, part_idx, st);
        default: return launch_fact_m<3, 6>(G, T, Jprev, part_val, part_idx, st);
    }
}

static inline bool is_column(const SdpTables& T) { return T.layout == SDP_LAYOUT_COLUMN_FACTORED; }
static inline bool is_tiled(const SdpTables& T) {
    return T.layout == SDP_LAYOUT_STATE_MINOR || T.layout == SDP_LAYOUT_STATE_MINOR_FACTORED || is_column(T);
}
static inline bool is_factored(const SdpTables& T) {
    return T.layout == SDP_LAYOUT_CONTROL_MINOR_FACTORED || T.layout == SDP_LAYOUT_STATE_MINOR_FACTORED ||
           is_column(T);
}
// layout CF, what the streaming pass needs on top of check_tables
static int check_column_stream(const SdpTables& T, const char* who) {
    if (!T.seg_begin || T.n_segs < 1 || T.n_segs > 0x7fffffffLL || !T.run_end)
        return fail(SDP_EINVAL, "%s: layout CF needs the CTA segments and column runs of the item list", who);
    if (!T.col_table || ((uintptr_t)T.col_table & 15))
        return fail(SDP_EINVAL, "%s: layout CF needs the 16-byte aligned column-table scratch", who);
    return SDP_OK;
}
// layout CF, combine pass: the view must be one band (whole rows, 32 per tile of a column)
static int check_column_band(const SdpTables& T, const char* who) {
    if (T.pos_row ? (T.n_states / T.n_cols > (int64_t)T.tiles_per_col * 32)
                  : ((T.n_states / T.n_cols + 31) / 32 != T.tiles_per_col))
        return fail(SDP_EINVAL, "%s: layout CF: the combine pass takes one band of rows at a time", who);
    return SDP_OK;
}
static int check_tables(const SdpTables& T, const char* who) {
    if (T.W < 1 || T.W > 4096 || T.n_states < 0 || T.n_items < 0)
        return fail(SDP_EINVAL, "%s: bad sizes", who);
    if (T.n_states == 0) return SDP_OK;
    if (!T.cell || !T.lam || !T.g || !T.items || !T.item_begin || (T.expect && !T.p))
        return fail(SDP_EINVAL, "%s: NULL pointer in tables", who);
    if ((T.lam_plane & 3) || ((uintptr_t)T.cell & 15) || ((uintptr_t)T.lam & 15) || ((uintptr_t)T.g & 15))
        return fail(SDP_EINVAL, "%s: tables must be 16-byte aligned, lam_plane % 4 == 0", who);
    if (T.layout < SDP_LAYOUT_CONTROL_MINOR || T.layout > SDP_LAYOUT_COLUMN_FACTORED)
        return fail(SDP_EINVAL, "%s: unknown table layout", who);
    if (is_tiled(T) && !T.U)
        return fail(SDP_EINVAL, "%s: layout B needs the per-state control counts", who);
    if (is_factored(T)) {
        if (T.g_per_w || !T.cell_w || !T.lam_w)
            return fail(SDP_EINVAL, "%s: factored tables need g per (x,u) and a w-part", who);
        if ((T.layout == SDP_LAYOUT_STATE_MINOR_FACTORED || is_column(T)) && T.W > SDP_FACTORED_MAX_W_REG)
            return fail(SDP_EINVAL, "%s: layouts BF / CF support at most 9 perturbation nodes", who);
        if ((T.layout == SDP_LAYOUT_STATE_MINOR_FACTORED || is_column(T)) && T.expect && !T.p_host)
            return fail(SDP_EINVAL, "%s: layouts BF / CF need p_host (host copy of the probabilities)", who);
        if (is_column(T)) {
            if (T.u_mask != 1)
                return fail(SDP_EINVAL, "%s: layout CF needs u_mask == 1 (axis 0 follows the control)", who);
            if (T.n_cols < 1 || T.tiles_per_col < 1 || T.n_states % T.n_cols != 0)
                return fail(SDP_EINVAL, "%s: layout CF: the shard must be whole rows of axis 0", who);
        }
        if (T.layout == SDP_LAYOUT_CONTROL_MINOR_FACTORED && T.W > 128)
            return fail(SDP_EINVAL, "%s: layout AF supports at most 128 perturbation nodes", who);
    }
    if (T.n_items / 8 + 1 > 0x7fffffffLL) return fail(SDP_EINVAL, "%s: too many items", who);
    return SDP_OK;
}

extern "C" int sdp_sweep_partials(const SdpGrid* grid, const SdpTables* tab, const double* J_prev,
                                  double* part_val, int32_t* part_idx, void* stream) {
    GridT<double> G;
    int rc = make_grid<double>(grid, &G, nullptr);
    if (rc) return rc;
    if (!tab) return fail(SDP_EINVAL, "%s", "sdp_sweep: tables is NULL");
    const SdpTables& T = *tab;
    rc = check_tables(T, "sdp_sweep");
    if (rc) return rc;
    if (T.n_states == 0 || T.n_items == 0) return SDP_OK;
    if (!J_prev || !part_val || !part_idx) return fail(SDP_EINVAL, "%s", "sdp_sweep: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (is_factored(T)) {
        rc = check_factored_args(grid->d, T.W, T.u_mask, "sdp_sweep");
        if (rc) return rc;
        if (T.layout == SDP_LAYOUT_COLUMN_FACTORED) {
            rc = check_column_stream(T, "sdp_sweep");
            if (rc) return rc;
            return grid->d == 2 ? launch_fact_column<2>(G, T, J_prev, part_val, part_idx, st)
                                : launch_fact_column<3>(G, T, J_prev, part_val, part_idx, st);
        }
        return grid->d == 2 ? launch_fact<2>(G, T, J_prev, part_val, part_idx, st)
                            : launch_fact<3>(G, T, J_prev, part_val, part_idx, st);
    }
    switch (grid->d) {
        case 1: return launch_sweep<1>(G, T, J_prev, part_val, part_idx, st);
        case 2: return launch_sweep<2>(G, T, J_prev, part_val, part_idx, st);
        case 3: return launch_sweep<3>(G, T, J_prev, part_val, part_idx, st);
        default: return launch_sweep<4>(G, T, J_prev, part_val, part_idx, st);
    }
}

extern "C" int sdp_column_table(const SdpGrid* grid, const SdpTables* tab, const double* J_prev, void* stream) {
    GridT<double> G;
    int rc = make_grid<double>(grid, &G, nullptr);
    if (rc) return rc;
    if (!tab) return fail(SDP_EINVAL, "%s", "sdp_column_table: tables is NULL");
    const SdpTables& T = *tab;
    rc = check_tables(T, "sdp_column_table");
    if (rc) return rc;
    if (!is_column(T)) return fail(SDP_EINVAL, "%s", "sdp_column_table: the tables are not in layout CF");
    if (T.n_states == 0 || T.n_items == 0) return SDP_OK;
    rc = check_factored_args(grid->d, T.W, T.u_mask, "sdp_column_table");
    if (!rc) rc = check_column_stream(T, "sdp_column_table");
    if (rc) return rc;
    if (!J_prev) return fail(SDP_EINVAL, "%s", "sdp_column_table: NULL pointer");
    if ((T.col_pairs ? SDP_COLUMN_PITCH2(G.order[0], T.W) : SDP_COLUMN_PITCH(G.order[0], T.W)) * 8 > SDP_COLUMN_MAX_SMEM_BYTES)
        return fail(SDP_EINVAL, "%s", "sdp_column_table: the column table does not fit shared memory");
    cudaStream_t st = (cudaStream_t)stream;
    return grid->d == 2 ? launch_column_table<2>(G, T, J_prev, st) : launch_column_table<3>(G, T, J_prev, st);
}

// (layout CF: the transposing combine kernel lives with the peer-memory code below)
static void launch_combine_column_local(const SdpTables& T, const double* part_val, const int32_t* part_idx,
                                        double* J_out, int32_t* argmin_out, cudaStream_t st);

extern "C" int sdp_sweep_finalize(const SdpTables* tab, const double* part_val,
                                  const int32_t* part_idx, double* J_out, int32_t* argmin_out,
                                  void* stream) {
    if (!tab) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize: tables is NULL");
    const SdpTables& T = *tab;
    int rc = check_tables(T, "sdp_sweep_finalize");
    if (rc) return rc;
    if (T.n_states == 0) return SDP_OK;
    if (is_column(T) && (rc = check_column_band(T, "sdp_sweep_finalize"))) return rc;
    if (!part_val || !part_idx || !J_out || !argmin_out)
        return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned blocks = (unsigned)((T.n_states + 255) / 256);
    if (is_column(T))
        launch_combine_column_local(T, part_val, part_idx, J_out, argmin_out, st);
    else if (is_tiled(T))
        k_sweep_finalize_tiled<<<blocks, 256, 0, st>>>(T.n_states, T.item_begin, part_val, part_idx, J_out, argmin_out,
                                                       0, T.tiles_per_col);
    else
        k_sweep_finalize<<<blocks, 256, 0, st>>>(T.n_states, T.item_begin, part_val, part_idx, J_out, argmin_out);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

extern "C" int sdp_sweep(const SdpGrid* grid, const SdpTables* tab, const double* J_prev,
                         double* part_val, int32_t* part_idx, double* J_out, int32_t* argmin_out,
                         void* stream) {
    int rc = sdp_sweep_partials(grid, tab, J_prev, part_val, part_idx, stream);
    if (rc) return rc;
    return sdp_sweep_finalize(tab, part_val, part_idx, J_out, argmin_out, stream);
}

// ---------------------------------------------------------------------------
// Multi-GPU: fused combine + all-gather over peer memory, flag barrier
// ---------------------------------------------------------------------------
// Publish: every CTA fences its peer stores (system scope), the last CTA to arrive
// bumps the rank's epoch and lanes 0..world-1 release it into the flag arrays of all
// ranks IN PARALLEL (one st.release.sys each: a loop in one thread would pay one
// NVLink round trip per peer, 8 in a row on a full box).  Called by all threads.
__device__ __forceinline__ void publish_epoch(const PeersDev& P, int dbg = 0) {
    __shared__ unsigned long long e_sh;
    __shared__ int last_sh;
    // ONE system-scope fence per CTA, by the thread that signals, after the CTA barrier: the
    // barrier orders the peer stores of all the CTA's threads before it and the fence is
    // cumulative (the pattern of a grid-wide barrier).  A fence in every thread was measured at
    // 33 us per launch on 2 and on 8 GPUs alike (the MEMBAR.SYS of the 32 warps of a CTA take
    // turns), four times the stores themselves.
    __syncthreads();
    if (threadIdx.x == 0) {
        if (!(dbg & 2)) __threadfence_system();
        const unsigned int prev = atomicAdd(P.done, 1u);
        last_sh = (prev == gridDim.x - 1);
        if (last_sh) {
            __threadfence();
            *P.done = 0;
            e_sh = *P.epoch + 1;
            *P.epoch = e_sh;
        }
    }
    __syncthreads();
    if (last_sh && threadIdx.x < P.world) {
        if (dbg & 4) *(volatile unsigned long long*)(P.flags[threadIdx.x] + P.rank) = e_sh;
        else st_release_sys(P.flags[threadIdx.x] + P.rank, e_sh);
    }
}

// per-state combine of the partial minima; J is stored into every rank's buffer
template <bool TILED>
__global__ void __launch_bounds__(256)
k_sweep_finalize_p2p(int64_t n_states, const int64_t* __restrict__ item_begin,
                     const double* __restrict__ part_val, const int32_t* __restrict__ part_idx,
                     int32_t* __restrict__ argmin_out, PeersDev P, int64_t state_begin,
                     int n_cols, int tiles_per_col) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_states) {
        int64_t unit = i;
        int lane = 0;
        if (TILED) tile_of_state(i, n_cols, tiles_per_col, unit, lane);
        const int width = TILED ? 32 : 1;
        double bv = CUDART_INF;
        int bi = INT_MAX;
        for (int64_t k = item_begin[unit]; k < item_begin[unit + 1]; ++k) {
            const double v = part_val[k * width + lane];
            const int ix = part_idx[k * width + lane];
            if (better(v, ix, bv, bi)) { bv = v; bi = ix; }
        }
        argmin_out[i] = bi;
#pragma unroll
        for (int r = 0; r < SDP_MAX_PEERS; ++r)
            if (r < P.world) P.J[r][state_begin + i] = bv;
        if (P.A[0]) {
#pragma unroll
            for (int r = 0; r < SDP_MAX_PEERS; ++r)
                if (r < P.world) P.A[r][state_begin + i] = bi;
        }
    }
    // publish: every CTA fences its peer stores, the last one to finish releases the epoch
    publish_epoch(P);
}

__global__ void k_p2p_wait(PeersDev P, unsigned long long timeout_ns) {
    const int t = threadIdx.x;
    if (t < P.world) {
        const unsigned long long e = *P.epoch;
        wait_flag(P.flags[P.rank] + t, e, timeout_ns);
    }
}

__global__ void k_p2p_barrier(PeersDev P, unsigned long long timeout_ns) {
    __shared__ unsigned long long e_sh;
    if (threadIdx.x == 0) {
        e_sh = *P.epoch + 1;
        *P.epoch = e_sh;
        __threadfence_system();
    }
    __syncthreads();
    const int t = threadIdx.x;
    if (t < P.world) {
        st_release_sys(P.flags[t] + P.rank, e_sh);
        wait_flag(P.flags[P.rank] + t, e_sh, timeout_ns);
    }
}

// Layout CF combine, both sides coalesced.  The partial minima of a tile are 32 lanes = 32
// consecutive ROWS of one column, the value function is C-order (columns fastest): a thread
// per state in grid order (k_sweep_finalize_tiled) reads every partial from another cache
// line - measured 35 us per sweep for the 125 000 states of one rank of eight, five times the
// peer stores themselves.  Here a CTA owns 32 rows x 32 columns of a band: warp w combines
// the items of column c0 + w (lanes = rows: one contiguous 256-byte read per item), the block
// transposes through shared memory, then warp w stores row r0 + w (lanes = columns: 256
// contiguous bytes into the local buffer, or into every rank's buffer over NVLink).
// State (row, col) of the band goes to J[j_offset + row * j_pitch + col] and to
// argmin_out[row * n_cols + col].  P.world == 0: local store into J_out, no epoch.
// value of control axis c at index idx of a grid of m points on [a, b]: the reference's
// np.linspace arithmetic (stodynprog.py:458, numpy's linspace: step = delta/div, y = idx*step + a,
// last point forced to b; one point: the middle)
__device__ __forceinline__ double control_axis_value(int m, int idx, double a, double b) {
    if (m == 1) return div_(add_(a, b), 2.0);
    if (idx == m - 1) return b;
    const double div = (double)(m - 1);
    const double delta = sub_(b, a);
    const double step = div_(delta, div);
    if (step == 0.0) return add_(mul_(div_((double)idx, div), delta), a);
    return add_(mul_((double)idx, step), a);
}

// optional tail of the CF combine: the argmin of every state mapped to control VALUES (K3 fused;
// lo / hi / npts / pol indexed by grid state like J_out).  nc == 0: off.
struct PolMap {
    int nc;
    const double* lo;
    const double* hi;
    const int32_t* npts;
    double* pol;
};

__global__ void __launch_bounds__(1024)
k_combine_column(int n_rows, int n_cols, int tiles_per_col, int col_blocks,
                 const int64_t* __restrict__ item_begin, const double* __restrict__ part_val,
                 const int32_t* __restrict__ part_idx, double* __restrict__ J_out,
                 int32_t* __restrict__ argmin_out, PeersDev P, int64_t j_offset, int64_t j_pitch, int dbg,
                 const int32_t* __restrict__ pos_row, int64_t a_offset, int64_t a_pitch, PolMap M) {
    __shared__ double v_sh[32][33];
    __shared__ int i_sh[32][33];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ty = blockIdx.x / col_blocks;                 // tile (32 rows) of the band
    cudaGridDependencySynchronize();       // (programmatic dependent launch: the sweep's partial minima)
    const int c0 = (blockIdx.x - ty * col_blocks) * 32;
    if (n_rows > 0) {
        const int c = c0 + warp;
        if (c < n_cols) {
            const int64_t tile = (int64_t)c * tiles_per_col + ty;
            double bv = CUDART_INF;
            int bi = INT_MAX;
            // (the partial minima of four items in flight at a time, compared in item order)
            const int64_t k1 = item_begin[tile + 1];
            for (int64_t k = item_begin[tile]; k < k1; k += 4) {
                double v[4];
                int ix[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int64_t kk = (k + u < k1) ? k + u : k1 - 1;
                    v[u] = part_val[kk * 32 + lane];
                    ix[u] = part_idx[kk * 32 + lane];
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (k + u < k1 && better(v[u], ix[u], bv, bi)) { bv = v[u]; bi = ix[u]; }
            }
            v_sh[lane][warp] = bv;
            i_sh[lane][warp] = bi;
        }
    }
    __syncthreads();
    if (n_rows > 0) {
        // (two rows per lane: position ty*32 + warp of the column holds row pos_row[...], -1 = padding)
        const int r = pos_row ? pos_row[ty * 32 + warp] : ty * 32 + warp, c = c0 + lane;
        if (r >= 0 && r < n_rows && c < n_cols) {
            const double bv = v_sh[warp][lane];
            argmin_out[a_offset + (int64_t)r * a_pitch + c] = i_sh[warp][lane];
            const int64_t g = j_offset + (int64_t)r * j_pitch + c;
            if (P.world == 0) {
                J_out[g] = bv;
                if (M.nc > 0) {
                    // (same arithmetic as k_policy_values)
                    long long rem = i_sh[warp][lane];
                    for (int k = M.nc - 1; k >= 0; --k) {
                        const int m = M.npts[g * M.nc + k];
                        const int idx = (int)(rem % m);
                        rem /= m;
                        M.pol[g * M.nc + k] = control_axis_value(m, idx, M.lo[g * M.nc + k], M.hi[g * M.nc + k]);
                    }
                }
            } else {
#pragma unroll
                for (int q = 0; q < SDP_MAX_PEERS; ++q)
                    if (q < P.world && (!(dbg & 1) || q == P.rank)) P.J[q][g] = bv;
                if (P.A[0]) {
                    // the argmin travels with J: every rank then holds the whole policy and can
                    // map and copy out any part of it (results fanned out over all PCIe links)
                    const int bi = i_sh[warp][lane];
#pragma unroll
                    for (int q = 0; q < SDP_MAX_PEERS; ++q)
                        if (q < P.world && (!(dbg & 1) || q == P.rank)) P.A[q][g] = bi;
                }
            }
        }
    }
    if (P.world > 0) publish_epoch(P, dbg);
}

// launch of the above for one band of layout CF
static void launch_combine_column(const SdpTables& T, const double* part_val, const int32_t* part_idx,
                                  double* J_out, int32_t* argmin_out, const PeersDev& P,
                                  int64_t j_offset, int64_t j_pitch, cudaStream_t st,
                                  int64_t a_offset = 0, int64_t a_pitch = -1, const PolMap* map = nullptr) {
    PolMap M;
    memset(&M, 0, sizeof(M));
    if (map) M = *map;
    if (a_pitch < 0) a_pitch = T.n_cols;       // (the argmin stays local: state r*n_cols + c of the shard)
    const int n_rows = T.n_cols > 0 ? (int)(T.n_states / T.n_cols) : 0;
    const int col_blocks = T.n_cols > 0 ? (T.n_cols + 31) / 32 : 1;
    unsigned blocks = (unsigned)col_blocks * (unsigned)(T.pos_row ? T.tiles_per_col : (n_rows + 31) / 32);
    if (blocks == 0 || n_rows == 0) blocks = 1;       // (an empty shard still publishes its epoch)
    launch_pdl(k_combine_column, dim3(blocks), dim3(1024), 0, st, n_rows, T.n_cols, T.tiles_per_col, col_blocks,
               T.item_begin, part_val, part_idx, J_out, argmin_out, P, j_offset, j_pitch,
               tuning().dbg_exchange, T.pos_row, a_offset, a_pitch, M);
}

static void launch_combine_column_local(const SdpTables& T, const double* part_val, const int32_t* part_idx,
                                        double* J_out, int32_t* argmin_out, cudaStream_t st) {
    PeersDev none;
    memset(&none, 0, sizeof(none));
    launch_combine_column(T, part_val, part_idx, J_out, argmin_out, none, 0, T.n_cols, st);
}

static int make_peers(const SdpPeers* p, PeersDev* out, const char* who) {
    if (!p) return fail(SDP_EINVAL, "%s: peers is NULL", who);
    if (p->world < 1 || p->world > SDP_MAX_PEERS || p->rank < 0 || p->rank >= p->world)
        return fail(SDP_EINVAL, "%s: bad world/rank", who);
    if (!p->epoch || !p->done) return fail(SDP_EINVAL, "%s: NULL epoch/done counter", who);
    out->world = p->world;
    out->rank = p->rank;
    for (int r = 0; r < SDP_MAX_PEERS; ++r) {
        out->J[r] = (r < p->world) ? p->J[r] : nullptr;
        out->A[r] = (r < p->world) ? p->A[r] : nullptr;
        out->flags[r] = (r < p->world) ? (unsigned long long*)p->flags[r] : nullptr;
        if (r < p->world && !p->flags[r]) return fail(SDP_EINVAL, "%s: NULL flag array", who);
    }
    out->epoch = (unsigned long long*)p->epoch;
    out->done = p->done;
    return SDP_OK;
}

extern "C" int sdp_sweep_finalize_p2p(const SdpTables* tab, const double* part_val,
                                      const int32_t* part_idx, int32_t* argmin_out,
                                      const SdpPeers* peers, int64_t state_begin, void* stream) {
    if (!tab) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_p2p: tables is NULL");
    const SdpTables& T = *tab;
    int rc = check_tables(T, "sdp_sweep_finalize_p2p");
    if (rc) return rc;
    if (is_column(T) && T.n_states > 0 && (rc = check_column_band(T, "sdp_sweep_finalize_p2p"))) return rc;
    PeersDev P;
    rc = make_peers(peers, &P, "sdp_sweep_finalize_p2p");
    if (rc) return rc;
    for (int r = 0; r < P.world; ++r)
        if (!P.J[r]) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_p2p: NULL J buffer");
    if (state_begin < 0 || (T.n_states > 0 && (!part_val || !part_idx || !argmin_out)))
        return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_p2p: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    // at least one CTA even for an empty slab: the epoch must advance on every rank
    unsigned blocks = (unsigned)((T.n_states + 255) / 256);
    if (blocks == 0) blocks = 1;
    if (is_column(T) && T.n_states > 0)
        launch_combine_column(T, part_val, part_idx, nullptr, argmin_out, P, state_begin, T.n_cols, st);
    else if (is_tiled(T))
        k_sweep_finalize_p2p<true><<<blocks, 256, 0, st>>>(T.n_states, T.item_begin, part_val, part_idx, argmin_out, P, state_begin,
                                                           0, T.tiles_per_col);
    else
        k_sweep_finalize_p2p<false><<<blocks, 256, 0, st>>>(T.n_states, T.item_begin, part_val, part_idx, argmin_out, P, state_begin, 0, 0);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

extern "C" int sdp_sweep_finalize_p2p_cols(const SdpTables* tab, const double* part_val,
                                           const int32_t* part_idx, int32_t* argmin_out,
                                           const SdpPeers* peers, int64_t glob_cols, int64_t col_begin,
                                           void* stream) {
    if (!tab) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_p2p_cols: tables is NULL");
    const SdpTables& T = *tab;
    int rc = check_tables(T, "sdp_sweep_finalize_p2p_cols");
    if (rc) return rc;
    if (!is_column(T)) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_p2p_cols: the tables are not in layout CF");
    if (T.n_states > 0 && (rc = check_column_band(T, "sdp_sweep_finalize_p2p_cols"))) return rc;
    PeersDev P;
    rc = make_peers(peers, &P, "sdp_sweep_finalize_p2p_cols");
    if (rc) return rc;
    for (int r = 0; r < P.world; ++r)
        if (!P.J[r]) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_p2p_cols: NULL J buffer");
    if (col_begin < 0 || glob_cols < col_begin + T.n_cols ||
        (T.n_states > 0 && (!part_val || !part_idx || !argmin_out)))
        return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_p2p_cols: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    // (an empty shard still launches one CTA: the epoch must advance on every rank)
    launch_combine_column(T, part_val, part_idx, nullptr, argmin_out, P, col_begin, glob_cols, st);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// The CF combine for the host path of one rank (sdp_sweep_finalize_cols): same tile of 32 rows x
// 32 columns transposed through shared memory as k_combine_column, but 128 threads and at most 32
// registers per thread, so that a CTA fits NEXT TO a resident CTA of the streaming kernel (768
// threads x 80 registers leave 4 096 registers per SM): the combine of one column piece then runs
// while the next piece is being swept on another stream, instead of waiting for an SM to drain,
// and the piece's results leave for the host that much earlier.  Maps the argmin to control
// values in the same pass (K3 fused).
__global__ void __launch_bounds__(128, 16)
k_combine_column_small(int n_rows, int n_cols, int tiles_per_col, int col_blocks,
                       const int64_t* __restrict__ item_begin, const double* __restrict__ part_val,
                       const int32_t* __restrict__ part_idx, double* __restrict__ J_out,
                       int32_t* __restrict__ argmin_out, int64_t offset, int64_t pitch,
                       const int32_t* __restrict__ pos_row, PolMap M) {
    __shared__ double v_sh[32][33];
    __shared__ int i_sh[32][33];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ty = blockIdx.x / col_blocks;                 // tile (32 rows) of the band
    const int c0 = (blockIdx.x - ty * col_blocks) * 32;
    // (few warps next to a busy streaming CTA: what counts is loads in flight - the item ranges of
    // the warp's 8 columns are fetched by 8 lanes at once, the partial minima 4 items at a time)
    long long b0 = 0, b1 = 0;
    if (lane < 8 && c0 + warp + 4 * lane < n_cols) {
        const int64_t tile = (int64_t)(c0 + warp + 4 * lane) * tiles_per_col + ty;
        b0 = item_begin[tile];
        b1 = item_begin[tile + 1];
    }
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
        const long long k0 = __shfl_sync(0xffffffffu, b0, j), k1 = __shfl_sync(0xffffffffu, b1, j);
        const int lc = warp + 4 * j;
        if (c0 + lc >= n_cols) break;
        double bv = CUDART_INF;
        int bi = INT_MAX;
        for (long long k = k0; k < k1; k += 4) {
            double v[4];
            int ix[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const long long kk = (k + u < k1) ? k + u : k1 - 1;
                v[u] = part_val[kk * 32 + lane];
                ix[u] = part_idx[kk * 32 + lane];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (k + u < k1 && better(v[u], ix[u], bv, bi)) { bv = v[u]; bi = ix[u]; }
        }
        v_sh[lane][lc] = bv;
        i_sh[lane][lc] = bi;
    }
    __syncthreads();
    const int c = c0 + lane;
    if (c >= n_cols) return;
    const int nc = M.nc;
    const double* __restrict__ lo = M.lo;
    const double* __restrict__ hi = M.hi;
    const int32_t* __restrict__ npts = M.npts;
    double* __restrict__ pol = M.pol;
#pragma unroll 2
    for (int lr = warp; lr < 32; lr += 4) {
        const int r = pos_row ? pos_row[ty * 32 + lr] : ty * 32 + lr;
        if (r < 0 || r >= n_rows) continue;
        const int64_t g = offset + (int64_t)r * pitch + c;
        const int bi = i_sh[lr][lane];
        J_out[g] = v_sh[lr][lane];
        argmin_out[g] = bi;
        unsigned rem = (unsigned)bi;          // (a flat index below 2^31)
        for (int k = nc - 1; k >= 0; --k) {
            const int m = npts[g * nc + k];
            const double a = lo[g * nc + k], b = hi[g * nc + k];
            const int idx = (int)(rem % (unsigned)m);
            rem /= (unsigned)m;
            pol[g * nc + k] = control_axis_value(m, idx, a, b);
        }
    }
}

// One rank, layout CF, results streamed by COLUMN pieces: the combine of the columns
// [col_begin, col_begin + tab->n_cols) of a grid of glob_cols columns (tab: a view whose item_begin
// starts at the first tile of col_begin).  J_out / argmin_out are whole-grid arrays in grid order;
// with nc > 0 the argmin is also mapped to control values (lo / hi / npts / pol whole-grid, [state][nc]).
// beside_sweep != 0: another piece is being swept meanwhile - launch the 128-thread variant whose CTAs
// fit next to the resident streaming CTAs; 0: the GPU is free, the 1024-thread variant is quicker.
extern "C" int sdp_sweep_finalize_cols(const SdpTables* tab, const double* part_val, const int32_t* part_idx,
                                       double* J_out, int32_t* argmin_out, int64_t glob_cols, int64_t col_begin,
                                       int32_t nc, const double* lo, const double* hi, const int32_t* npts,
                                       double* pol, int32_t beside_sweep, void* stream) {
    if (!tab) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_cols: tables is NULL");
    const SdpTables& T = *tab;
    int rc = check_tables(T, "sdp_sweep_finalize_cols");
    if (rc) return rc;
    if (!is_column(T)) return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_cols: the tables are not in layout CF");
    if (T.n_states == 0) return SDP_OK;
    if ((rc = check_column_band(T, "sdp_sweep_finalize_cols"))) return rc;
    if (col_begin < 0 || glob_cols < col_begin + T.n_cols || !part_val || !part_idx || !J_out || !argmin_out ||
        nc < 0 || (nc > 0 && (!lo || !hi || !npts || !pol)))
        return fail(SDP_EINVAL, "%s", "sdp_sweep_finalize_cols: bad arguments");
    PeersDev none;
    memset(&none, 0, sizeof(none));
    PolMap M;
    M.nc = nc; M.lo = lo; M.hi = hi; M.npts = npts; M.pol = pol;
    const int n_rows = (int)(T.n_states / T.n_cols);
    const int col_blocks = (T.n_cols + 31) / 32;
    const unsigned blocks = (unsigned)col_blocks * (unsigned)(T.pos_row ? T.tiles_per_col : (n_rows + 31) / 32);
    static bool carve_set = false;
    if (!carve_set && tuning().carveout) {
        cudaFuncSetAttribute(k_combine_column_small, cudaFuncAttributePreferredSharedMemoryCarveout,
                             cudaSharedmemCarveoutMaxShared);
        carve_set = true;
    }
    if (beside_sweep && tuning().small_combine)
        k_combine_column_small<<<blocks, 128, 0, (cudaStream_t)stream>>>(
            n_rows, T.n_cols, T.tiles_per_col, col_blocks, T.item_begin, part_val, part_idx, J_out, argmin_out,
            col_begin, glob_cols, T.pos_row, M);
    else
        launch_combine_column(T, part_val, part_idx, J_out, argmin_out, none, col_begin, glob_cols,
                              (cudaStream_t)stream, col_begin, glob_cols, &M);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// `height` rows of `width` bytes from src (pitch spitch) to dst (pitch dpitch), asynchronously on
// the stream; either side may be device or page-locked host memory (the column pieces of a result
// go to their place in the caller's C-order host arrays this way)
extern "C" int sdp_memcpy_2d(void* dst, int64_t dpitch, const void* src, int64_t spitch, int64_t width,
                             int64_t height, void* stream) {
    if (width < 0 || height < 0 || dpitch < width || spitch < width)
        return fail(SDP_EINVAL, "%s", "sdp_memcpy_2d: bad sizes");
    if (width == 0 || height == 0) return SDP_OK;
    if (!dst || !src) return fail(SDP_EINVAL, "%s", "sdp_memcpy_2d: NULL pointer");
    cudaError_t e = cudaMemcpy2DAsync(dst, (size_t)dpitch, src, (size_t)spitch, (size_t)width, (size_t)height,
                                      cudaMemcpyDefault, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(SDP_ECUDA, "sdp_memcpy_2d: %s", cudaGetErrorString(e));
    return SDP_OK;
}

extern "C" int sdp_p2p_wait(const SdpPeers* peers, void* stream) {
    PeersDev P;
    int rc = make_peers(peers, &P, "sdp_p2p_wait");
    if (rc) return rc;
    k_p2p_wait<<<1, 32, 0, (cudaStream_t)stream>>>(P, (unsigned long long)tuning().p2p_timeout_s * 1000000000ULL);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// n values of src (this rank's copy, device) starting at `offset` -> the same place of every
// OTHER rank's J buffer, then the epoch (follow with sdp_p2p_wait): the hand-over of an uploaded
// piece of J to the peers in one launch
__global__ void __launch_bounds__(256)
k_p2p_broadcast(const double* __restrict__ src, int64_t offset, int64_t n, PeersDev P) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = src[offset + i];
#pragma unroll
        for (int q = 0; q < SDP_MAX_PEERS; ++q)
            if (q < P.world && q != P.rank) P.J[q][offset + i] = v;
    }
    publish_epoch(P);
}

extern "C" int sdp_p2p_broadcast(const double* src, int64_t offset, int64_t n, const SdpPeers* peers, void* stream) {
    PeersDev P;
    int rc = make_peers(peers, &P, "sdp_p2p_broadcast");
    if (rc) return rc;
    if (offset < 0 || n < 0 || (n > 0 && !src)) return fail(SDP_EINVAL, "%s", "sdp_p2p_broadcast: bad arguments");
    for (int r = 0; r < P.world; ++r)
        if (!P.J[r]) return fail(SDP_EINVAL, "%s", "sdp_p2p_broadcast: NULL J buffer");
    int64_t blocks = (n + 255) / 256;
    if (blocks < 1) blocks = 1;            // (an empty piece still publishes the epoch)
    if (blocks > 148 * 4) blocks = 148 * 4;
    k_p2p_broadcast<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(src, offset, n, P);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

extern "C" int sdp_sweep_partials_after(const SdpGrid* grid, const SdpTables* tab, const double* J_prev,
                                        double* part_val, int32_t* part_idx, const SdpPeers* wait_for,
                                        void* stream) {
    PeersDev P;
    int rc = make_peers(wait_for, &P, "sdp_sweep_partials_after");
    if (rc) return rc;
    const bool fold = tab && tab->layout == SDP_LAYOUT_COLUMN_FACTORED && tuning().col_prepass &&
                      !tab->col_table_ready && tab->n_states > 0 && tab->n_items > 0;
    if (!fold) {
        // no kernel of this layout can carry the wait: a separate launch, as sdp_p2p_wait
        k_p2p_wait<<<1, 32, 0, (cudaStream_t)stream>>>(P, (unsigned long long)tuning().p2p_timeout_s * 1000000000ULL);
        SDP_LAUNCH_CHECK();
        return sdp_sweep_partials(grid, tab, J_prev, part_val, part_idx, stream);
    }
    g_wait_peers = &P;
    rc = sdp_sweep_partials(grid, tab, J_prev, part_val, part_idx, stream);
    if (g_wait_peers) {           // an argument check failed before the pre-pass was launched
        g_wait_peers = nullptr;
        if (!rc) rc = fail(SDP_EINVAL, "%s", "sdp_sweep_partials_after: the wait was not enqueued");
    }
    return rc;
}

extern "C" int sdp_p2p_barrier(const SdpPeers* peers, void* stream) {
    PeersDev P;
    int rc = make_peers(peers, &P, "sdp_p2p_barrier");
    if (rc) return rc;
    k_p2p_barrier<<<1, 32, 0, (cudaStream_t)stream>>>(P, (unsigned long long)tuning().p2p_timeout_s * 1000000000ULL);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K1': fixed-policy backup. One thread per state, tables are [w][n_states]
// planes so that adjacent threads read adjacent entries.
// ---------------------------------------------------------------------------
// one fixed-policy backup: sum_w p_w * (g + J(f(x, pol(x), w)))   (stodynprog.py:755,757);
// entry w of the state sits at index w*stride of its arrays
template <int D>
__device__ __forceinline__ double policy_backup(const GridT<double>& G, int W, int g_per_w,
                                                const double* __restrict__ p,
                                                const int32_t* __restrict__ cell,
                                                const double* __restrict__ lam, int64_t lam_plane,
                                                const double* __restrict__ g, int64_t stride,
                                                const double* __restrict__ J_in) {
    double acc = 0.0;
    double gv = g_per_w ? 0.0 : g[0];
    for (int w = 0; w < W; ++w) {
        const int64_t off = (int64_t)w * stride;
        double l[D];
#pragma unroll
        for (int k = 0; k < D; ++k) l[k] = lam[(int64_t)k * lam_plane + off];
        if (g_per_w) gv = g[off];
        double v = Lerp<double, D, 0>::eval(J_in, cell[off], G.stride, l);
        acc = add_(acc, mul_(add_(gv, v), p[w]));
    }
    return acc;
}

// the table entries of the reference state of relative DP (device pointers)
struct RefState {
    const int32_t* cell;
    const double* lam;
    int64_t lam_plane;
    const double* g;
    int64_t stride;
    double* hist;       // J_ref of this iteration is written here (by block 0)
};

// Relative DP (stodynprog.py:760-762: J_ref[k] = J_pol[ref_ind]; J_pol -= J_ref[k]) is
// fused into the backup: thread 0 of every block recomputes the backup of the reference
// state (the same operations in the same order, hence the same bits as the thread that
// owns that state) and the block subtracts it - one launch per iteration instead of
// three (backup, pick, subtract) in a loop that is launch-latency bound.
template <int D, bool REL>
__global__ void __launch_bounds__(256)
k_policy_eval(GridT<double> G, int W, int g_per_w, const double* __restrict__ p,
              const int32_t* __restrict__ cell, const double* __restrict__ lam, int64_t lam_plane,
              const double* __restrict__ g, int64_t n_states, const double* __restrict__ J_in,
              double* __restrict__ J_out, RefState R) {
    __shared__ double ref_sh;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double acc = 0.0;
    if (i < n_states)
        acc = policy_backup<D>(G, W, g_per_w, p, cell + i, lam + i, lam_plane, g + i, n_states, J_in);
    if (REL) {
        if (threadIdx.x == 0) {
            ref_sh = policy_backup<D>(G, W, g_per_w, p, R.cell, R.lam, R.lam_plane, R.g, R.stride, J_in);
            if (blockIdx.x == 0) R.hist[0] = ref_sh;
        }
        __syncthreads();
        acc = sub_(acc, ref_sh);
    }
    if (i < n_states) J_out[i] = acc;
}

// Fixed-policy backup fused with the all-gather: the new value of every state of the
// slab goes straight into every rank's J buffer (peer-mapped pointers), the last CTA
// publishes the epoch - the same protocol as k_sweep_finalize_p2p.
template <int D, bool REL>
__global__ void __launch_bounds__(256)
k_policy_eval_p2p(GridT<double> G, int W, int g_per_w, const double* __restrict__ p,
                  const int32_t* __restrict__ cell, const double* __restrict__ lam, int64_t lam_plane,
                  const double* __restrict__ g, int64_t n_states, const double* __restrict__ J_in,
                  PeersDev P, int64_t state_begin, RefState R) {
    __shared__ double ref_sh;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double acc = 0.0;
    if (i < n_states)
        acc = policy_backup<D>(G, W, g_per_w, p, cell + i, lam + i, lam_plane, g + i, n_states, J_in);
    if (REL) {
        if (threadIdx.x == 0) {
            ref_sh = policy_backup<D>(G, W, g_per_w, p, R.cell, R.lam, R.lam_plane, R.g, R.stride, J_in);
            if (blockIdx.x == 0) R.hist[0] = ref_sh;
        }
        __syncthreads();
        acc = sub_(acc, ref_sh);
    }
    if (i < n_states) {
#pragma unroll
        for (int r = 0; r < SDP_MAX_PEERS; ++r)
            if (r < P.world) P.J[r][state_begin + i] = acc;
    }
    publish_epoch(P);
}

__global__ void k_pick(const double* __restrict__ J, int64_t idx, double* __restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) out[0] = J[idx];
}
__global__ void __launch_bounds__(256)
k_sub_scalar(double* __restrict__ J, int64_t n, const double* __restrict__ ref) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) J[i] = sub_(J[i], ref[0]);
}

static int rel_shift_launch(double* J, int64_t n, int64_t ref_index, double* ref_out, cudaStream_t st) {
    k_pick<<<1, 32, 0, st>>>(J, ref_index, ref_out);
    SDP_LAUNCH_CHECK();
    k_sub_scalar<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(J, n, ref_out);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

extern "C" int sdp_rel_shift(double* J, int64_t n, int64_t ref_index, double* ref_out, void* stream) {
    if (!J || !ref_out || n <= 0 || ref_index < 0 || ref_index >= n)
        return fail(SDP_EINVAL, "%s", "sdp_rel_shift: bad arguments");
    return rel_shift_launch(J, n, ref_index, ref_out, (cudaStream_t)stream);
}

extern "C" int sdp_policy_eval(const SdpGrid* grid, int32_t W, int32_t g_per_w, const double* p,
                               const int32_t* cell, const double* lam, int64_t lam_plane,
                               const double* g, int64_t n_states, int64_t state_begin, int64_t n_grid,
                               double* J_a, double* J_b, int32_t n_iter, int32_t rel_dp,
                               int64_t ref_index, double* J_ref_hist, void* stream) {
    GridT<double> G;
    int64_t ng = 0;
    int rc = make_grid<double>(grid, &G, &ng);
    if (rc) return rc;
    if (W < 1 || n_states < 0 || n_iter < 0 || n_grid != ng || state_begin < 0 ||
        state_begin + n_states > n_grid)
        return fail(SDP_EINVAL, "%s", "sdp_policy_eval: bad sizes");
    if (n_iter == 0 || n_states == 0) return SDP_OK;
    if (!p || !cell || !lam || !g || !J_a || !J_b) return fail(SDP_EINVAL, "%s", "sdp_policy_eval: NULL pointer");
    if (rel_dp && (!J_ref_hist || n_states != n_grid || ref_index < 0 || ref_index >= n_grid))
        return fail(SDP_EINVAL, "%s", "sdp_policy_eval: rel_dp needs the whole grid in one shard and a J_ref_hist buffer");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned blocks = (unsigned)((n_states + 255) / 256);
    double* in = J_a;
    double* out = J_b;
    RefState R = {nullptr, nullptr, 0, nullptr, 0, nullptr};
    if (rel_dp) {
        // the reference state belongs to this shard (whole grid): its entries are in the tables
        const int64_t ir = ref_index - state_begin;
        R.cell = cell + ir; R.lam = lam + ir; R.lam_plane = lam_plane; R.g = g + ir; R.stride = n_states;
    }
    for (int it = 0; it < n_iter; ++it) {
        double* o = out + state_begin;
        if (rel_dp) {
            R.hist = J_ref_hist + it;
            switch (grid->d) {
                case 1: k_policy_eval<1, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
                case 2: k_policy_eval<2, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
                case 3: k_policy_eval<3, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
                default: k_policy_eval<4, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
            }
        } else {
            switch (grid->d) {
                case 1: k_policy_eval<1, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
                case 2: k_policy_eval<2, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
                case 3: k_policy_eval<3, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
                default: k_policy_eval<4, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, in, o, R); break;
            }
        }
        SDP_LAUNCH_CHECK();
        double* t = in; in = out; out = t;
    }
    return SDP_OK;
}

extern "C" int sdp_policy_eval_p2p(const SdpGrid* grid, int32_t W, int32_t g_per_w, const double* p,
                                   const int32_t* cell, const double* lam, int64_t lam_plane,
                                   const double* g, int64_t n_states, int64_t state_begin,
                                   int64_t n_grid, const double* J_in, const SdpPeers* peers,
                                   const int32_t* ref_cell, const double* ref_lam,
                                   const double* ref_g, double* J_ref_out, void* stream) {
    GridT<double> G;
    int64_t ng = 0;
    int rc = make_grid<double>(grid, &G, &ng);
    if (rc) return rc;
    if (W < 1 || n_states < 0 || n_grid != ng || state_begin < 0 || state_begin + n_states > n_grid)
        return fail(SDP_EINVAL, "%s", "sdp_policy_eval_p2p: bad sizes");
    PeersDev P;
    rc = make_peers(peers, &P, "sdp_policy_eval_p2p");
    if (rc) return rc;
    for (int r = 0; r < P.world; ++r)
        if (!P.J[r]) return fail(SDP_EINVAL, "%s", "sdp_policy_eval_p2p: NULL J buffer");
    if (!J_in || (n_states > 0 && (!p || !cell || !lam || !g)))
        return fail(SDP_EINVAL, "%s", "sdp_policy_eval_p2p: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned blocks = (unsigned)((n_states + 255) / 256);
    if (blocks == 0) blocks = 1;      // the epoch must advance on every rank, even for an empty slab
    if (ref_cell) {
        // relative DP: every rank holds a copy of the reference state's W entries ([w], stride 1)
        if (!ref_lam || !ref_g || !J_ref_out || !p)
            return fail(SDP_EINVAL, "%s", "sdp_policy_eval_p2p: incomplete reference-state arguments");
        RefState R = {ref_cell, ref_lam, (int64_t)W, ref_g, 1, J_ref_out};
        switch (grid->d) {
            case 1: k_policy_eval_p2p<1, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
            case 2: k_policy_eval_p2p<2, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
            case 3: k_policy_eval_p2p<3, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
            default: k_policy_eval_p2p<4, true><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
        }
    } else {
        RefState R = {nullptr, nullptr, 0, nullptr, 0, nullptr};
        switch (grid->d) {
            case 1: k_policy_eval_p2p<1, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
            case 2: k_policy_eval_p2p<2, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
            case 3: k_policy_eval_p2p<3, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
            default: k_policy_eval_p2p<4, false><<<blocks, 256, 0, st>>>(G, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J_in, P, state_begin, R); break;
        }
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K1'': forward (adjoint) operator of a fixed policy, mu <- P^T mu (include/sdp_b200.h).
// New feature: the reference only simulates trajectories (storage_control.py:217,246).
// Build: CSR by destination from the [w][n] policy-table planes of K1'.  Steps: a gather, one
// warp per destination row; no floating-point atomics, every sum in a fixed association.
// ---------------------------------------------------------------------------
#define SDP_FWD_ROWS_PER_CTA 256   // one tile of the cost / residual partial sums

static inline int64_t align256(int64_t b) { return (b + 255) & ~(int64_t)255; }

// destination of corner eps of base cell b: bit k of eps is the corner along axis k
__device__ __forceinline__ int fwd_dest(const GridT<double>& G, int d, int b, int eps) {
    int y = b;
#pragma unroll
    for (int k = 0; k < SDP_MAX_D; ++k)
        if (k < d && ((eps >> k) & 1)) y += G.stride[k];
    return y;
}

// one thread per (x, w) table entry e = w*n + x: count the 2^d destinations
__global__ void __launch_bounds__(256)
k_fwd_count(GridT<double> G, int d, int64_t nw, const int32_t* __restrict__ cell, int32_t* __restrict__ counts) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nw) return;
    const int b = cell[e];
    for (int eps = 0; eps < (1 << d); ++eps) atomicAdd(counts + fwd_dest(G, d, b, eps), 1);
}

// same walk: every entry lands at row_ptr[y] + (a cursor of row y) with its source key
// (x*W + w)*2^d + eps; the order inside a row is fixed afterwards by sorting the keys
__global__ void __launch_bounds__(256)
k_fwd_fill(GridT<double> G, int d, int W, int64_t n, const int32_t* __restrict__ cell,
           const int64_t* __restrict__ row_ptr, int32_t* __restrict__ cursor, int32_t* __restrict__ keys) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * W) return;
    const int64_t w = e / n, x = e - w * n;
    const int b = cell[e];
    const int key0 = (int)((x * W + w) << d);
    for (int eps = 0; eps < (1 << d); ++eps) {
        const int y = fwd_dest(G, d, b, eps);
        keys[row_ptr[y] + atomicAdd(cursor + y, 1)] = key0 + eps;
    }
}

// key -> (source state, coefficient p_w * f_0 * ... * f_{d-1}, left to right); in place on src
__global__ void __launch_bounds__(256)
k_fwd_coef(int d, int W, int64_t n, int64_t nnz, const double* __restrict__ p, const double* __restrict__ lam,
           int64_t lam_plane, int32_t* __restrict__ src, double* __restrict__ coef) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    const int key = src[j];
    const int eps = key & ((1 << d) - 1);
    const int xw = key >> d;
    const int x = xw / W, w = xw - x * W;
    const int64_t e = (int64_t)w * n + x;
    double c = p[w];
#pragma unroll
    for (int k = 0; k < SDP_MAX_D; ++k) {
        if (k < d) {
            const double l = lam[(int64_t)k * lam_plane + e];
            c = mul_(c, ((eps >> k) & 1) ? l : sub_(1.0, l));
        }
    }
    src[j] = x;
    coef[j] = c;
}

// g_bar(x) = sum_w p_w * g(x, w), accumulated in w order from 0
__global__ void __launch_bounds__(256)
k_fwd_gbar(int W, int g_per_w, int64_t n, const double* __restrict__ p, const double* __restrict__ g,
           double* __restrict__ gbar) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    double acc = 0.0;
    for (int w = 0; w < W; ++w) acc = add_(acc, mul_(p[w], g[g_per_w ? (int64_t)w * n + x : x]));
    gbar[x] = acc;
}

// pieces per row: ceil(len / SDP_FWD_PIECE) for rows longer than one piece, 0 otherwise
__global__ void __launch_bounds__(256)
k_fwd_piece_count(int64_t n, const int64_t* __restrict__ row_ptr, int32_t* __restrict__ counts) {
    const int64_t y = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (y > n) return;
    if (y == n) { counts[n] = 0; return; }
    const int64_t len = row_ptr[y + 1] - row_ptr[y];
    counts[y] = len > SDP_FWD_PIECE ? (int32_t)((len + SDP_FWD_PIECE - 1) / SDP_FWD_PIECE) : 0;
}

__global__ void __launch_bounds__(256)
k_fwd_piece_fill(int64_t n, const int64_t* __restrict__ piece_first, int32_t* __restrict__ piece_row) {
    const int64_t y = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= n) return;
    for (int64_t q = piece_first[y]; q < piece_first[y + 1]; ++q) piece_row[q] = (int32_t)y;
}

// sum of coef[e] * mu[src[e]] over [begin, end) by a team of TEAM lanes: lane-strided in index
// order, then a butterfly inside the team (every lane of the team ends with the same bits: IEEE
// addition is commutative).  TEAM is a constant of the operator, not of the launch.
template <int TEAM>
__device__ __forceinline__ double fwd_segment(const int32_t* __restrict__ src, const double* __restrict__ coef,
                                              const double* __restrict__ mu, int64_t begin, int64_t end,
                                              int tl) {
    double acc = 0.0;
#pragma unroll 4
    for (int64_t e = begin + tl; e < end; e += TEAM)
        acc = add_(acc, mul_(__ldcs(coef + e), __ldg(mu + __ldcs(src + e))));
#pragma unroll
    for (int o = TEAM / 2; o >= 1; o >>= 1) acc = add_(acc, __shfl_xor_sync(0xffffffffu, acc, o));
    return acc;
}

// one warp per piece of a long row
__global__ void __launch_bounds__(256)
k_fwd_pieces(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ src, const double* __restrict__ coef,
             const int64_t* __restrict__ piece_first, const int32_t* __restrict__ piece_row, int64_t n_pieces,
             const double* __restrict__ mu, double* __restrict__ piece_val) {
    const int lane = threadIdx.x & 31;
    const int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= n_pieces) return;
    const int y = piece_row[q];
    const int64_t begin = row_ptr[y] + (q - piece_first[y]) * SDP_FWD_PIECE;
    const int64_t end = min(begin + SDP_FWD_PIECE, row_ptr[y + 1]);
    const double v = fwd_segment<32>(src, coef, mu, begin, end, lane);
    if (lane == 0) piece_val[q] = v;
}

// the row pass: CTA t owns rows [256t, 256t+256), warp i rows 256t + 32i + j, j = 0..31.  The
// warp loads the bounds of its 32 rows once (lane j: row j), then sums them SDP_FWD_TEAMS rows at
// a time, a team of 32/SDP_FWD_TEAMS lanes per row (rows hold n*W*2^d/n entries on average: 36 for
// W = 9, d = 2), so that several rows' loads are in flight per warp.  Lane j collects row j's value,
// stores it (coalesced) and forms the cost / residual terms of its row; partials of the tile:
// part[t] = sum mu_in*g_bar, part[n_tiles + t] = sum |mu_out - mu_in|
#define SDP_FWD_TEAMS 4
__global__ void __launch_bounds__(SDP_FWD_ROWS_PER_CTA)
k_fwd_rows(int64_t n, const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ src,
           const double* __restrict__ coef, const int64_t* __restrict__ piece_first,
           const double* __restrict__ piece_val, const double* __restrict__ gbar,
           const double* __restrict__ mu_in, double* __restrict__ mu_out, double* __restrict__ hist_out,
           double* __restrict__ part, int64_t n_tiles) {
    constexpr int TEAM = 32 / SDP_FWD_TEAMS;
    __shared__ double sh[2][SDP_FWD_ROWS_PER_CTA / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int team = lane / TEAM, tl = lane % TEAM;
    const int64_t base = (int64_t)blockIdx.x * SDP_FWD_ROWS_PER_CTA + warp * 32;
    const int64_t y = base + lane;
    int64_t r0 = 0, r1 = 0, q0 = 0, q1 = 0;
    if (y < n) { r0 = row_ptr[y]; r1 = row_ptr[y + 1]; q0 = piece_first[y]; q1 = piece_first[y + 1]; }
    double mine = 0.0;
#pragma unroll 1
    for (int j0 = 0; j0 < 32; j0 += SDP_FWD_TEAMS) {
        const int j = j0 + team;
        const int64_t b = __shfl_sync(0xffffffffu, r0, j), e = __shfl_sync(0xffffffffu, r1, j);
        const int64_t p0 = __shfl_sync(0xffffffffu, q0, j), p1 = __shfl_sync(0xffffffffu, q1, j);
        double v;
        if (p0 == p1) {
            v = fwd_segment<TEAM>(src, coef, mu_in, b, e, tl);          // empty beyond n: b == e == 0
        } else {
            double acc = 0.0;                 // pieces of a long row, in piece order
            for (int64_t q = p0 + tl; q < p1; q += TEAM) acc = add_(acc, piece_val[q]);
#pragma unroll
            for (int o = TEAM / 2; o >= 1; o >>= 1) acc = add_(acc, __shfl_xor_sync(0xffffffffu, acc, o));
            v = acc;
        }
        const double got = __shfl_sync(0xffffffffu, v, ((lane - j0) & (SDP_FWD_TEAMS - 1)) * TEAM);
        if (lane >= j0 && lane < j0 + SDP_FWD_TEAMS) mine = got;
    }
    double c = 0.0, r = 0.0;
    if (y < n) {
        mu_out[y] = mine;
        if (hist_out) hist_out[y] = mine;
        const double m = mu_in[y];
        c = mul_(m, gbar[y]);
        r = fabs(sub_(mine, m));
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        c = add_(c, __shfl_xor_sync(0xffffffffu, c, o));
        r = add_(r, __shfl_xor_sync(0xffffffffu, r, o));
    }
    if (lane == 0) { sh[0][warp] = c; sh[1][warp] = r; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double cs = 0.0, rs = 0.0;
        for (int i = 0; i < SDP_FWD_ROWS_PER_CTA / 32; ++i) { cs = add_(cs, sh[0][i]); rs = add_(rs, sh[1][i]); }
        part[blockIdx.x] = cs;
        part[n_tiles + blockIdx.x] = rs;
    }
}

// one CTA: thread t sums the tiles t, t+256, ... in order, then a fixed tree over the threads
__global__ void __launch_bounds__(256)
k_fwd_reduce(const double* __restrict__ part, int64_t n_tiles, double* __restrict__ cost_out,
             double* __restrict__ resid_out) {
    __shared__ double sc[256], sr[256];
    double c = 0.0, r = 0.0;
    for (int64_t t = threadIdx.x; t < n_tiles; t += 256) {
        c = add_(c, part[t]);
        r = add_(r, part[n_tiles + t]);
    }
    sc[threadIdx.x] = c;
    sr[threadIdx.x] = r;
    __syncthreads();
    for (int s = 128; s >= 1; s >>= 1) {
        if (threadIdx.x < s) {
            sc[threadIdx.x] = add_(sc[threadIdx.x], sc[threadIdx.x + s]);
            sr[threadIdx.x] = add_(sr[threadIdx.x], sr[threadIdx.x + s]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        cost_out[0] = sc[0];
        if (resid_out) resid_out[0] = sr[0];
    }
}

// byte offsets inside the build scratch: counts / cursors int32 [n+1], keys int32 [nnz], cub's
// temporary storage (the larger of the scans' and the segmented sort's)
struct FwdScratch {
    int64_t keys_off, temp_off, temp_bytes, total;
};

static int fwd_sizes(int d, int W, int64_t n, int64_t* nnz, FwdScratch* S) {
    if (d < 1 || d > SDP_MAX_D || W < 1 || n < 1) return fail(SDP_EINVAL, "%s", "sdp_forward: bad sizes");
    const int64_t z = n * (int64_t)W << d;
    if (z >= (int64_t)INT_MAX || n >= (int64_t)INT_MAX)
        return fail(SDP_EINVAL, "%s", "sdp_forward: n*W*2^d must stay below 2^31");
    size_t scan_b = 0, sort_b = 0;
    SDP_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, scan_b, (const int32_t*)nullptr, (int64_t*)nullptr,
                                                 (int)(n + 1)));
    SDP_CUDA_CHECK(cub::DeviceSegmentedSort::SortKeys(nullptr, sort_b, (const int32_t*)nullptr, (int32_t*)nullptr,
                                                      z, n, (const int64_t*)nullptr, (const int64_t*)nullptr));
    *nnz = z;
    S->keys_off = align256(4 * (n + 1));
    S->temp_off = S->keys_off + align256(4 * z);
    S->temp_bytes = (int64_t)(scan_b > sort_b ? scan_b : sort_b);
    S->total = S->temp_off + align256(S->temp_bytes);
    return SDP_OK;
}

static int64_t fwd_max_pieces(int64_t nnz) { return 2 * (nnz / SDP_FWD_PIECE) + 1; }

extern "C" int sdp_forward_sizes(int32_t d, int32_t W, int64_t n, int64_t* nnz, int64_t* max_pieces,
                                 int64_t* build_scratch_bytes, int64_t* step_scratch_doubles) {
    if (!nnz || !max_pieces || !build_scratch_bytes || !step_scratch_doubles)
        return fail(SDP_EINVAL, "%s", "sdp_forward_sizes: NULL pointer");
    FwdScratch S;
    int rc = fwd_sizes(d, W, n, nnz, &S);
    if (rc) return rc;
    *max_pieces = fwd_max_pieces(*nnz);
    *build_scratch_bytes = S.total;
    *step_scratch_doubles = *max_pieces + 2 * ((n + SDP_FWD_ROWS_PER_CTA - 1) / SDP_FWD_ROWS_PER_CTA);
    return SDP_OK;
}

extern "C" int sdp_forward_build(const SdpGrid* grid, int32_t W, int32_t g_per_w, const double* p,
                                 const int32_t* cell, const double* lam, int64_t lam_plane, const double* g,
                                 const SdpForwardOp* op, void* scratch, int64_t scratch_bytes, void* stream) {
    GridT<double> G;
    int64_t ng = 0;
    int rc = make_grid<double>(grid, &G, &ng);
    if (rc) return rc;
    if (!op) return fail(SDP_EINVAL, "%s", "sdp_forward_build: NULL op");
    const int d = grid->d;
    const int64_t n = op->n;
    int64_t nnz = 0;
    FwdScratch S;
    if (n != ng) return fail(SDP_EINVAL, "%s", "sdp_forward_build: op->n is not the grid size");
    rc = fwd_sizes(d, W, n, &nnz, &S);
    if (rc) return rc;
    if (op->nnz != nnz || op->max_pieces < fwd_max_pieces(nnz) || lam_plane < W * n || scratch_bytes < S.total)
        return fail(SDP_EINVAL, "%s", "sdp_forward_build: buffer sizes do not match sdp_forward_sizes");
    if (!p || !cell || !lam || !g || !scratch || !op->row_ptr || !op->src || !op->coef || !op->gbar ||
        !op->piece_first || !op->piece_row)
        return fail(SDP_EINVAL, "%s", "sdp_forward_build: NULL pointer");
    if (((uintptr_t)scratch) & 255) return fail(SDP_EINVAL, "%s", "sdp_forward_build: scratch not 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char* sb = (char*)scratch;
    int32_t* counts = (int32_t*)sb;
    int32_t* keys = (int32_t*)(sb + S.keys_off);
    void* temp = sb + S.temp_off;
    size_t temp_bytes = (size_t)S.temp_bytes;
    const int64_t nw = n * W;
    const unsigned bw = (unsigned)((nw + 255) / 256);
    SDP_CUDA_CHECK(cudaMemsetAsync(counts, 0, 4 * (n + 1), st));
    k_fwd_count<<<bw, 256, 0, st>>>(G, d, nw, cell, counts);
    SDP_LAUNCH_CHECK();
    SDP_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, (const int32_t*)counts, op->row_ptr,
                                                 (int)(n + 1), st));
    SDP_CUDA_CHECK(cudaMemsetAsync(counts, 0, 4 * (n + 1), st));
    k_fwd_fill<<<bw, 256, 0, st>>>(G, d, W, n, cell, op->row_ptr, counts, keys);
    SDP_LAUNCH_CHECK();
    temp_bytes = (size_t)S.temp_bytes;
    SDP_CUDA_CHECK(cub::DeviceSegmentedSort::SortKeys(temp, temp_bytes, (const int32_t*)keys, op->src, nnz, n,
                                                      (const int64_t*)op->row_ptr, (const int64_t*)op->row_ptr + 1, st));
    k_fwd_coef<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(d, W, n, nnz, p, lam, lam_plane, op->src, op->coef);
    SDP_LAUNCH_CHECK();
    const unsigned bn = (unsigned)((n + 256) / 256);
    k_fwd_gbar<<<bn, 256, 0, st>>>(W, g_per_w, n, p, g, op->gbar);
    SDP_LAUNCH_CHECK();
    k_fwd_piece_count<<<bn, 256, 0, st>>>(n, op->row_ptr, counts);
    SDP_LAUNCH_CHECK();
    temp_bytes = (size_t)S.temp_bytes;
    SDP_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, (const int32_t*)counts, op->piece_first,
                                                 (int)(n + 1), st));
    k_fwd_piece_fill<<<bn, 256, 0, st>>>(n, op->piece_first, op->piece_row);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

extern "C" int sdp_forward_steps(const SdpForwardOp* op, double* mu_a, double* mu_b, int32_t n_steps,
                                 double* cost_out, double* resid_out, double* hist, double* scratch,
                                 void* stream) {
    if (!op || n_steps < 0 || op->n < 1 || op->n_pieces < 0 || op->n_pieces > op->max_pieces)
        return fail(SDP_EINVAL, "%s", "sdp_forward_steps: bad sizes");
    if (!mu_a || !mu_b || (n_steps > 0 && (!cost_out || !scratch || !op->row_ptr || !op->src || !op->coef ||
                                           !op->gbar || !op->piece_first || (op->n_pieces && !op->piece_row))))
        return fail(SDP_EINVAL, "%s", "sdp_forward_steps: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = op->n;
    if (hist) SDP_CUDA_CHECK(cudaMemcpyAsync(hist, mu_a, 8 * n, cudaMemcpyDeviceToDevice, st));
    const int64_t n_tiles = (n + SDP_FWD_ROWS_PER_CTA - 1) / SDP_FWD_ROWS_PER_CTA;
    double* piece_val = scratch;
    double* part = scratch + op->max_pieces;
    const double* in = mu_a;
    double* out = mu_b;
    for (int k = 0; k < n_steps; ++k) {
        if (op->n_pieces > 0) {
            k_fwd_pieces<<<(unsigned)((op->n_pieces + 7) / 8), 256, 0, st>>>(
                op->row_ptr, op->src, op->coef, op->piece_first, op->piece_row, op->n_pieces, in, piece_val);
            SDP_LAUNCH_CHECK();
        }
        k_fwd_rows<<<(unsigned)n_tiles, SDP_FWD_ROWS_PER_CTA, 0, st>>>(
            n, op->row_ptr, op->src, op->coef, op->piece_first, piece_val, op->gbar, in, out,
            hist ? hist + (int64_t)(k + 1) * n : nullptr, part, n_tiles);
        SDP_LAUNCH_CHECK();
        k_fwd_reduce<<<1, 256, 0, st>>>(part, n_tiles, cost_out + k, k + 1 == n_steps ? resid_out : nullptr);
        SDP_LAUNCH_CHECK();
        const double* t = in;
        in = out;
        out = const_cast<double*>(t);
    }
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K1''': sample paths of a fixed policy's chain (include/sdp_b200.h).  New feature: the
// reference simulates the policy on the host (storage_control.py:217,246).  One thread per path,
// its state in registers; a transition reads one packed (x, w) record, one 32-byte sector for
// d <= 2.  Random numbers are counter-based (Philox-4x32-10), so a path's results depend only on
// (seed, path, tables), not on the launch shape.
// ---------------------------------------------------------------------------
#define SDP_CHAIN_THREADS 256

// Philox-4x32-10 (Salmon et al., SC'11; the Random123 reference): 10 rounds, key bumped between them
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        if (i) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    }
    return c;
}

// a double in [0, 1) from two words: the top 53 bits of (lo | hi << 32), exact
__device__ __forceinline__ double chain_u01(uint32_t lo, uint32_t hi) {
    return (double)((((uint64_t)hi << 32) | lo) >> 11) * 0x1p-53;
}

// first index j < len with t < C[j], len - 1 if none (C non-decreasing)
__device__ __forceinline__ int chain_search(const double* C, int len, double t) {
    int lo = 0, hi = len - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (t < C[mid]) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

template <int D>
__global__ void __launch_bounds__(256)
k_chain_pack(int W, int g_per_w, int64_t n, const int32_t* __restrict__ cell, const double* __restrict__ lam,
             int64_t lam_plane, const double* __restrict__ g, double* __restrict__ rec) {
    constexpr int REC = SDP_CHAIN_REC(D);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * W) return;
    double r[REC];
    r[0] = __longlong_as_double((long long)(uint32_t)cell[e]);
#pragma unroll
    for (int k = 0; k < D; ++k) r[1 + k] = lam[(int64_t)k * lam_plane + e];
    r[1 + D] = g[g_per_w ? e : e % n];
    if (REC > D + 2) r[REC - 1] = 0.0;
    double2* out = reinterpret_cast<double2*>(rec + e * REC);
#pragma unroll
    for (int j = 0; j < REC / 2; ++j) out[j] = make_double2(r[2 * j], r[2 * j + 1]);
}

// one thread per path.  Per global step s: record, target test, then the transition out of s
template <int D>
__global__ void __launch_bounds__(1024)
k_chain_sample(GridT<double> G, int W, const double* __restrict__ cdf, const double* __restrict__ rec, int64_t n,
               int64_t M, int n_steps, uint32_t step0, uint2 key, int fresh, const double* __restrict__ start_cdf,
               const uint32_t* __restrict__ target, const int32_t* __restrict__ rec_steps, int n_rec,
               int32_t* __restrict__ state, double* __restrict__ total, int32_t* __restrict__ hit,
               int32_t* __restrict__ rec_out, unsigned long long* __restrict__ counters) {
    constexpr int REC = SDP_CHAIN_REC(D);
    extern __shared__ double chain_cdf[];
    __shared__ unsigned int chain_cnt[2];
    for (int j = threadIdx.x; j < W; j += blockDim.x) chain_cdf[j] = cdf[j];
    if (threadIdx.x < 2) chain_cnt[threadIdx.x] = 0u;
    __syncthreads();
    const double cmax = chain_cdf[W - 1];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int n_clamped = 0, n_nan = 0;
    if (i < M) {
        const uint32_t path = (uint32_t)i;
        int x, h;
        double acc;
        if (fresh) {
            acc = 0.0;
            h = -1;
            if (start_cdf) {
                const uint4 r = philox4x32_10(make_uint4(path, SDP_CHAIN_INIT_STEP, 0u, 0u), key);
                const double t = chain_u01(r.x, r.y) * __ldg(start_cdf + n - 1);
                int lo = 0, hi = (int)n - 1;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (t < __ldg(start_cdf + mid)) hi = mid;
                    else lo = mid + 1;
                }
                x = lo;
            } else {
                x = state[i];
            }
        } else {
            x = state[i];
            acc = total[i];
            h = hit[i];
        }
        int r = 0;
        while (r < n_rec && (uint32_t)__ldg(rec_steps + r) < step0) ++r;
#pragma unroll 1
        for (int k = 0;; ++k) {
            const uint32_t s = step0 + (uint32_t)k;
            if (r < n_rec && (uint32_t)__ldg(rec_steps + r) == s) rec_out[(int64_t)r++ * M + i] = x;
            if (target && h < 0 && ((__ldg(target + (x >> 5)) >> (x & 31)) & 1u)) h = (int)s;
            if (k == n_steps) break;
            const uint4 r0 = philox4x32_10(make_uint4(path, s, 0u, 0u), key);
            const int w = chain_search(chain_cdf, W, chain_u01(r0.x, r0.y) * cmax);
            const double2* R = reinterpret_cast<const double2*>(rec + ((int64_t)w * n + x) * REC);
            double q[REC];
#pragma unroll
            for (int j = 0; j < REC / 2; ++j) {
                const double2 t = __ldg(R + j);
                q[2 * j] = t.x;
                q[2 * j + 1] = t.y;
            }
            double v[D];
            v[0] = chain_u01(r0.z, r0.w);
            if (D >= 2) {
                const uint4 r1 = philox4x32_10(make_uint4(path, s, 1u, 0u), key);
                v[1 % D] = chain_u01(r1.x, r1.y);
                if (D >= 3) v[2 % D] = chain_u01(r1.z, r1.w);
            }
            if (D >= 4) {
                const uint4 r2 = philox4x32_10(make_uint4(path, s, 2u, 0u), key);
                v[3 % D] = chain_u01(r2.x, r2.y);
            }
            int y = (int)(uint32_t)__double_as_longlong(q[0]);
            bool clamped = false, nan = false;
#pragma unroll
            for (int kk = 0; kk < D; ++kk) {
                double l = q[1 + kk];
                if (l != l) {
                    nan = true;
                    continue;
                }
                if (l < 0.0) { l = 0.0; clamped = true; }
                else if (l > 1.0) { l = 1.0; clamped = true; }
                if (v[kk] < l) y += G.stride[kk];
            }
            acc = add_(acc, q[1 + D]);
            n_clamped += clamped;
            n_nan += nan;
            x = y;
        }
        state[i] = x;
        total[i] = acc;
        hit[i] = h;
    }
    n_clamped = __reduce_add_sync(0xffffffffu, n_clamped);
    n_nan = __reduce_add_sync(0xffffffffu, n_nan);
    if ((threadIdx.x & 31) == 0 && (n_clamped | n_nan)) {
        atomicAdd(chain_cnt, n_clamped);
        atomicAdd(chain_cnt + 1, n_nan);
    }
    __syncthreads();
    if (threadIdx.x == 0 && (chain_cnt[0] | chain_cnt[1])) {
        atomicAdd(counters, (unsigned long long)chain_cnt[0]);
        atomicAdd(counters + 1, (unsigned long long)chain_cnt[1]);
    }
}

extern "C" int sdp_chain_pack(const SdpGrid* grid, int32_t W, int32_t g_per_w, const int32_t* cell,
                              const double* lam, int64_t lam_plane, const double* g, int64_t n, double* rec,
                              void* stream) {
    GridT<double> G;
    int64_t ng = 0;
    int rc = make_grid<double>(grid, &G, &ng);
    if (rc) return rc;
    if (W < 1 || n != ng || lam_plane < W * n || n * W >= (int64_t)INT_MAX)
        return fail(SDP_EINVAL, "%s", "sdp_chain_pack: bad sizes");
    if (!cell || !lam || !g || !rec) return fail(SDP_EINVAL, "%s", "sdp_chain_pack: NULL pointer");
    if (((uintptr_t)rec) & 15) return fail(SDP_EINVAL, "%s", "sdp_chain_pack: rec not 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned b = (unsigned)((n * W + 255) / 256);
    switch (grid->d) {
        case 1: k_chain_pack<1><<<b, 256, 0, st>>>(W, g_per_w, n, cell, lam, lam_plane, g, rec); break;
        case 2: k_chain_pack<2><<<b, 256, 0, st>>>(W, g_per_w, n, cell, lam, lam_plane, g, rec); break;
        case 3: k_chain_pack<3><<<b, 256, 0, st>>>(W, g_per_w, n, cell, lam, lam_plane, g, rec); break;
        default: k_chain_pack<4><<<b, 256, 0, st>>>(W, g_per_w, n, cell, lam, lam_plane, g, rec); break;
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

extern "C" int sdp_chain_sample(const SdpGrid* grid, int32_t W, const double* cdf, const double* rec, int64_t M,
                                int32_t n_steps, int64_t step0, uint64_t seed, int32_t fresh,
                                const double* start_cdf, const uint32_t* target, const int32_t* rec_steps,
                                int32_t n_rec, int32_t* state, double* total, int32_t* hit, int32_t* rec_out,
                                unsigned long long* counters, void* stream) {
    GridT<double> G;
    int64_t n = 0;
    int rc = make_grid<double>(grid, &G, &n);
    if (rc) return rc;
    if (W < 1 || M < 1 || M >= ((int64_t)1 << 31) || n_steps < 0 || step0 < 0 || n_rec < 0 ||
        step0 + n_steps >= (int64_t)SDP_CHAIN_INIT_STEP || n * W >= (int64_t)INT_MAX)
        return fail(SDP_EINVAL, "%s", "sdp_chain_sample: bad sizes");
    if ((size_t)W * 8 > 48 * 1024) return fail(SDP_EINVAL, "%s", "sdp_chain_sample: W > 6144 nodes");
    if (!cdf || !rec || !state || !total || !hit || !counters || (n_rec && (!rec_steps || !rec_out)))
        return fail(SDP_EINVAL, "%s", "sdp_chain_sample: NULL pointer");
    if (((uintptr_t)rec) & 15) return fail(SDP_EINVAL, "%s", "sdp_chain_sample: rec not 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int threads = tuning().chain_threads ? tuning().chain_threads : SDP_CHAIN_THREADS;
    const unsigned blocks = (unsigned)((M + threads - 1) / threads);
    const size_t shm = (size_t)W * 8;
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
#define SDP_CHAIN_ARGS G, W, cdf, rec, n, M, n_steps, (uint32_t)step0, key, fresh, fresh ? start_cdf : nullptr, \
        target, rec_steps, n_rec, state, total, hit, rec_out, counters
    switch (grid->d) {
        case 1: k_chain_sample<1><<<blocks, threads, shm, st>>>(SDP_CHAIN_ARGS); break;
        case 2: k_chain_sample<2><<<blocks, threads, shm, st>>>(SDP_CHAIN_ARGS); break;
        case 3: k_chain_sample<3><<<blocks, threads, shm, st>>>(SDP_CHAIN_ARGS); break;
        default: k_chain_sample<4><<<blocks, threads, shm, st>>>(SDP_CHAIN_ARGS); break;
    }
#undef SDP_CHAIN_ARGS
    SDP_LAUNCH_CHECK();
    note_kernel("k_chain_sample<D=%d>, %d threads", grid->d, threads);
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K3: argmin index -> control values  u_grids[c].flatten()[ind_opt[c]]
// (stodynprog.py:686-689).  The control grid of a state is np.linspace(lo, hi,
// npts) - element i is i*step + lo with step = (hi-lo)/(npts-1) (true
// division), (i/div)*delta + lo when step == 0, and exactly `hi` for the last
// point - or the single centre point (lo+hi)/2 when npts == 1
// (stodynprog.py:449-458, numpy/_core/function_base.py linspace).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_policy_values(int64_t n, int nc, const double* __restrict__ lo, const double* __restrict__ hi,
                const int32_t* __restrict__ npts, const int32_t* __restrict__ argmin,
                double* __restrict__ pol) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long rem = argmin[i];
    for (int c = nc - 1; c >= 0; --c) {
        const int m = npts[i * nc + c];
        const int idx = (int)(rem % m);
        rem /= m;
        pol[i * nc + c] = control_axis_value(m, idx, lo[i * nc + c], hi[i * nc + c]);
    }
}

extern "C" int sdp_policy_values(int64_t n, int32_t nc, const double* lo, const double* hi,
                                 const int32_t* npts, const int32_t* argmin, double* pol,
                                 void* stream) {
    if (n < 0 || nc < 0) return fail(SDP_EINVAL, "%s", "sdp_policy_values: bad sizes");
    if (n == 0 || nc == 0) return SDP_OK;
    if (!lo || !hi || !npts || !argmin || !pol) return fail(SDP_EINVAL, "%s", "sdp_policy_values: NULL pointer");
    k_policy_values<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, nc, lo, hi, npts, argmin, pol);
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// sup-norm of the update
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_supnorm_diff(const double* __restrict__ a, const double* __restrict__ b, int64_t n,
               unsigned long long* __restrict__ out) {
    double m = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        double d = fabs(sub_(a[i], b[i]));
        if (d > m) m = d;  // NaN never compares greater: ignored
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        double o = __shfl_xor_sync(0xffffffffu, m, s);
        if (o > m) m = o;
    }
    // non-negative doubles order like their bit patterns
    if ((threadIdx.x & 31) == 0 && m > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

extern "C" int sdp_supnorm_diff(const double* a, const double* b, int64_t n, double* out, void* stream) {
    if (!out || n < 0 || (n > 0 && (!a || !b))) return fail(SDP_EINVAL, "%s", "sdp_supnorm_diff: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    SDP_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double), st));
    if (n == 0) return SDP_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    k_supnorm_diff<<<(unsigned)blocks, 256, 0, st>>>(a, b, n, reinterpret_cast<unsigned long long*>(out));
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K2: general multilinear interpolation, n_v value rows x n_s points
// ---------------------------------------------------------------------------
template <typename T, int D>
__global__ void __launch_bounds__(256)
k_interp(GridT<T> G, int64_t n_grid, int64_t n_v, const T* __restrict__ values, int64_t n_s,
         const T* __restrict__ s, T* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_s) return;
    int base = 0;
    T lam[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        int q;
        cell_1d<T>(s[(int64_t)k * n_s + i], G.smin[k], G.span[k], G.om1[k], G.order[k], q, lam[k]);
        base += q * G.stride[k];
    }
    for (int64_t v = 0; v < n_v; ++v)
        out[v * n_s + i] = Lerp<T, D, 0>::eval(values + v * n_grid, base, G.stride, lam);
}

template <typename T>
static int interp_impl(const SdpGrid* grid, int64_t n_v, const T* values, int64_t n_s, const T* s,
                       T* out, void* stream) {
    GridT<T> G;
    int64_t ng = 0;
    int rc = make_grid<T>(grid, &G, &ng);
    if (rc) return rc;
    if (n_v < 0 || n_s < 0) return fail(SDP_EINVAL, "%s", "sdp_interp: bad sizes");
    if (n_v == 0 || n_s == 0) return SDP_OK;
    if (!values || !s || !out) return fail(SDP_EINVAL, "%s", "sdp_interp: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned blocks = (unsigned)((n_s + 255) / 256);
    switch (grid->d) {
        case 1: k_interp<T, 1><<<blocks, 256, 0, st>>>(G, ng, n_v, values, n_s, s, out); break;
        case 2: k_interp<T, 2><<<blocks, 256, 0, st>>>(G, ng, n_v, values, n_s, s, out); break;
        case 3: k_interp<T, 3><<<blocks, 256, 0, st>>>(G, ng, n_v, values, n_s, s, out); break;
        default: k_interp<T, 4><<<blocks, 256, 0, st>>>(G, ng, n_v, values, n_s, s, out); break;
    }
    SDP_LAUNCH_CHECK();
    return SDP_OK;
}

// ---------------------------------------------------------------------------
// K2 on the host, for a handful of points.  The reference's simulation loops call the policy
// interpolant one scalar point at a time (examples/20 .../storage_control.py:217,246): through
// the GPU that is two PCIe crossings and a launch per point.  Same arithmetic as k_interp,
// operation for operation (x86 cvttsd2si cast semantics, true division, no contraction: the
// host pass is compiled with -ffp-contract=off), so both paths return the same bits.
// ---------------------------------------------------------------------------
static inline int host_trunc(double t) {
    if (!(t > -2147483649.0 && t < 2147483648.0)) return INT_MIN;
    return (int)t;
}
static inline int host_trunc(float t) {
    if (!(t >= -2147483648.0f && t < 2147483648.0f)) return INT_MIN;
    return (int)t;
}
static double host_lerp(const double* V, int base, const int* stride, const double* lam, int D, int K) {
    if (K == D) return V[base];
    const double a = host_lerp(V, base, stride, lam, D, K + 1);
    const double b = host_lerp(V, base + (K == D - 1 ? 1 : stride[K]), stride, lam, D, K + 1);
    const double oml = 1.0 - lam[K];
    const double x = oml * a, y = lam[K] * b;
    return x + y;
}
// fp32: the generated C of the reference evaluates (1.0 - lam)*a and the sums in double, the
// innermost lam*v product in float, one rounding to float at the end (see Lerp<float,...>)
static double host_lerp_f(const float* V, int base, const int* stride, const float* lam, int D, int K) {
    if (K == D - 1) {
        const float v0 = V[base], v1 = V[base + stride[K]];
        const float t2 = lam[K] * v1;
        const double x = (1.0 - (double)lam[K]) * (double)v0;
        return x + (double)t2;
    }
    const double a = host_lerp_f(V, base, stride, lam, D, K + 1);
    const double b = host_lerp_f(V, base + stride[K], stride, lam, D, K + 1);
    const double x = (1.0 - (double)lam[K]) * a, y = (double)lam[K] * b;
    return x + y;
}
template <typename T>
static int interp_host_impl(const SdpGrid* grid, int64_t n_v, const T* values, int64_t n_s, const T* s, T* out) {
    GridT<T> G;
    int64_t ng = 0;
    int rc = make_grid<T>(grid, &G, &ng);
    if (rc) return rc;
    if (n_v < 0 || n_s < 0) return fail(SDP_EINVAL, "%s", "sdp_interp_host: bad sizes");
    if (n_v == 0 || n_s == 0) return SDP_OK;
    if (!values || !s || !out) return fail(SDP_EINVAL, "%s", "sdp_interp_host: NULL pointer");
    const int D = grid->d;
    for (int64_t i = 0; i < n_s; ++i) {
        int base = 0;
        T lam[SDP_MAX_D];
        for (int k = 0; k < D; ++k) {
            const T d0 = s[(int64_t)k * n_s + i] - G.smin[k];
            const T sn = d0 / G.span[k];
            const T t = sn * G.om1[k];
            int q = host_trunc(t);
            q = q < G.order[k] - 2 ? q : G.order[k] - 2;
            q = q > 0 ? q : 0;
            lam[k] = t - (T)q;
            base += q * G.stride[k];
        }
        for (int64_t v = 0; v < n_v; ++v) {
            if (sizeof(T) == 8)
                out[v * n_s + i] = (T)host_lerp((const double*)(values + v * ng), base, G.stride, (const double*)lam, D, 0);
            else
                out[v * n_s + i] = (T)(float)host_lerp_f((const float*)(values + v * ng), base, G.stride, (const float*)lam, D, 0);
        }
    }
    return SDP_OK;
}
extern "C" int sdp_interp_host(const SdpGrid* grid, int64_t n_v, const double* values, int64_t n_s,
                               const double* s, double* out) {
    return interp_host_impl<double>(grid, n_v, values, n_s, s, out);
}
extern "C" int sdp_interp_host_f32(const SdpGrid* grid, int64_t n_v, const float* values, int64_t n_s,
                                   const float* s, float* out) {
    return interp_host_impl<float>(grid, n_v, values, n_s, s, out);
}

extern "C" int sdp_interp(const SdpGrid* grid, int64_t n_v, const double* values, int64_t n_s,
                          const double* s, double* out, void* stream) {
    return interp_impl<double>(grid, n_v, values, n_s, s, out, stream);
}
extern "C" int sdp_interp_f32(const SdpGrid* grid, int64_t n_v, const float* values, int64_t n_s,
                              const float* s, float* out, void* stream) {
    return interp_impl<float>(grid, n_v, values, n_s, s, out, stream);
}
