// gpa.cu -- bandwidth-bound kernels of the latent-GP target and gradient (src/GPA.jl).
//
//  * gpa_trmv: f = L v (unwhiten, GPA.jl:106) and w = L' g (the process block of dll, GPA.jl:200) on the resident factor.
//    One CTA per lower 128 x 128 tile of L writes its partial product; a second kernel adds the partials of every
//    output element in tile order.  No dependency chain, every summation order fixed: bitwise reproducible.
//  * gpa_row_scan: Z' of the closed-form reverse-mode Cholesky (DESIGN.md section 9.4).  Row b of Z' is a weighted prefix
//    sum along row b of W' = L^-T:  Z'[b,k] = w_k (sum_{l<k} v_l W'[b,l] + v_k W'[b,k] / 2).  Tile-parallel in three
//    launches: per-tile row sums, their exclusive prefix along each row (tile order), then the in-tile scans.
#include "gpa.cuh"

namespace {

constexpr int T = 128;
constexpr int NT = 256;

// linear index over the tiles (a, b), a >= b, of a triangle of tiles (row-major: (0,0), (1,0), (1,1), (2,0), ...)
__device__ __forceinline__ void tri_index(int lin, int& a, int& b) {
    a = (int)((sqrt(8.0 * (double)lin + 1.0) - 1.0) * 0.5);
    while (a * (a + 1) / 2 > lin) --a;
    while ((a + 1) * (a + 2) / 2 <= lin) ++a;
    b = lin - a * (a + 1) / 2;
}

// tile (bm, bn), bm >= bn, of L.  !TRANS: part[bn][bm*128 + r] = sum_c L[r,c] x[bn*128 + c]
//                                  TRANS: part[bm][bn*128 + c] = sum_r L[r,c] x[bm*128 + r]
template <bool TRANS>
__global__ void __launch_bounds__(NT) trmv_tile_kernel(const double* __restrict__ F, long long ld, long long Npad,
                                                       const double* __restrict__ x, double* __restrict__ part) {
    int bm, bn;
    tri_index(blockIdx.x, bm, bn);
    const bool diag = bm == bn;
    const double* tile = F + (long long)bm * T * ld + (long long)bn * T;
    if (!TRANS) {
        const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
        double xv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) xv[q] = x[(long long)bn * T + l + 32 * q];
#pragma unroll 4
        for (int rr = 0; rr < 16; ++rr) {
            const int r = w * 16 + rr;
            const double* row = tile + (long long)r * ld;
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int c = l + 32 * q;
                if (!diag || c <= r) s += row[c] * xv[q];       // the upper part of a diagonal tile is not L
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (l == 0) part[(long long)bn * Npad + (long long)bm * T + r] = s;
        }
    } else {
        __shared__ double sx[T], sh[T];
        if (threadIdx.x < T) sx[threadIdx.x] = x[(long long)bm * T + threadIdx.x];
        __syncthreads();
        const int c = threadIdx.x & (T - 1), h = threadIdx.x >> 7;
        double s = 0.0;
#pragma unroll 8
        for (int r = h * 64; r < h * 64 + 64; ++r)
            if (!diag || r >= c) s += tile[(long long)r * ld + c] * sx[r];
        if (h == 1) sh[c] = s;
        __syncthreads();
        if (h == 0) part[(long long)bm * Npad + (long long)bn * T + c] = s + sh[c];
    }
}

// out[i] = sum over the tiles of row-tile (or column-tile) i/128 of part, in tile order
template <bool TRANS>
__global__ void trmv_reduce_kernel(const double* __restrict__ part, long long Npad, double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Npad) return;
    const int t0 = (int)(i / T), nt = (int)(Npad / T);
    double s = 0.0;
    if (!TRANS) for (int t = 0; t <= t0; ++t) s += part[(long long)t * Npad + i];
    else        for (int t = t0; t < nt; ++t) s += part[(long long)t * Npad + i];
    out[i] = s;
}

// element (r, c) of the tile (bm, bn), bm <= bn, of W' (diagonal tiles: the clean upper-triangular DinvT)
__device__ __forceinline__ const double* wt_tile(const double* G, long long ld, const double* DinvT, int bm, int bn) {
    return bm == bn ? DinvT + (long long)bm * T * T : G + (long long)bm * T * ld + (long long)bn * T;
}

// pass 1: tsum[bn][bm*128 + r] = sum_c W'[bm*128 + r, bn*128 + c] v[bn*128 + c]  over the upper tiles bm <= bn
__global__ void __launch_bounds__(NT) scan_sums_kernel(const double* __restrict__ G, long long ld, const double* __restrict__ DinvT,
                                                       const double* __restrict__ v, long long Npad, double* __restrict__ tsum) {
    int bn, bm;
    tri_index(blockIdx.x, bn, bm);
    const double* tile = wt_tile(G, ld, DinvT, bm, bn);
    const long long ldt = bm == bn ? T : ld;
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    double vv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) vv[q] = v[(long long)bn * T + l + 32 * q];
#pragma unroll 4
    for (int rr = 0; rr < 16; ++rr) {
        const int r = w * 16 + rr;
        const double* row = tile + (long long)r * ldt;
        double s = row[l] * vv[0] + row[l + 32] * vv[1] + row[l + 64] * vv[2] + row[l + 96] * vv[3];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (l == 0) tsum[(long long)bn * Npad + (long long)bm * T + r] = s;
    }
}

// pass 2: exclusive prefix of the tile sums along every row (tile order), in place
__global__ void scan_prefix_kernel(double* __restrict__ tsum, long long Npad) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Npad) return;
    const int nt = (int)(Npad / T);
    double acc = 0.0;
    for (int t = (int)(i / T); t < nt; ++t) {
        const double x = tsum[(long long)t * Npad + i];
        tsum[(long long)t * Npad + i] = acc;
        acc += x;
    }
}

// pass 3: in-tile scans (one warp per row, 32-wide shuffle scans carried across the four column quarters)
__global__ void __launch_bounds__(NT) scan_apply_kernel(const double* __restrict__ G, long long ld, const double* __restrict__ DinvT,
                                                        const double* __restrict__ v, const double* __restrict__ w,
                                                        long long Npad, const double* __restrict__ tsum,
                                                        double* __restrict__ F, double* __restrict__ Zd) {
    int bn, bm;
    tri_index(blockIdx.x, bn, bm);
    const bool diag = bm == bn;
    const double* tile = wt_tile(G, ld, DinvT, bm, bn);
    const long long ldt = diag ? T : ld;
    double* out = diag ? Zd + (long long)bm * T * T : F + (long long)bm * T * ld + (long long)bn * T;
    const int warp = threadIdx.x >> 5, l = threadIdx.x & 31;
    double vv[4], ww[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) { vv[q] = v[(long long)bn * T + l + 32 * q]; ww[q] = w[(long long)bn * T + l + 32 * q]; }
#pragma unroll 1
    for (int rr = 0; rr < 16; ++rr) {
        const int r = warp * 16 + rr;
        const double* row = tile + (long long)r * ldt;
        double carry = tsum[(long long)bn * Npad + (long long)bm * T + r];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double x = row[l + 32 * q] * vv[q];
            double inc = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double y = __shfl_up_sync(0xffffffffu, inc, o);
                if (l >= o) inc += y;
            }
            double exc = __shfl_up_sync(0xffffffffu, inc, 1);
            if (l == 0) exc = 0.0;
            out[(long long)r * ldt + l + 32 * q] = ww[q] * (carry + exc + 0.5 * x);
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
    }
}

}  // namespace

cudaError_t gpa_trmv(const double* F, int64_t ld, int64_t Npad, bool trans, const double* x, double* part, double* out,
                     cudaStream_t st, int64_t* launches) {
    const int nt = (int)(Npad / T);
    const unsigned tiles = (unsigned)(nt * (nt + 1) / 2);
    const unsigned rb = (unsigned)((Npad + NT - 1) / NT);
    if (trans) {
        trmv_tile_kernel<true><<<tiles, NT, 0, st>>>(F, ld, Npad, x, part);
        trmv_reduce_kernel<true><<<rb, NT, 0, st>>>(part, Npad, out);
    } else {
        trmv_tile_kernel<false><<<tiles, NT, 0, st>>>(F, ld, Npad, x, part);
        trmv_reduce_kernel<false><<<rb, NT, 0, st>>>(part, Npad, out);
    }
    *launches += 2;
    return cudaGetLastError();
}

cudaError_t gpa_row_scan(const double* G, int64_t ld, const double* DinvT, const double* v, const double* w, int64_t Npad,
                         double* tsum, double* F, double* Zd, cudaStream_t st, int64_t* launches) {
    const int nt = (int)(Npad / T);
    const unsigned tiles = (unsigned)(nt * (nt + 1) / 2);
    scan_sums_kernel<<<tiles, NT, 0, st>>>(G, ld, DinvT, v, Npad, tsum);
    scan_prefix_kernel<<<(unsigned)((Npad + NT - 1) / NT), NT, 0, st>>>(tsum, Npad);
    scan_apply_kernel<<<tiles, NT, 0, st>>>(G, ld, DinvT, v, w, Npad, tsum, F, Zd);
    *launches += 3;
    return cudaGetLastError();
}
