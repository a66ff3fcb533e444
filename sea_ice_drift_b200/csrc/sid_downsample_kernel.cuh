// sid_downsample_kernel.cuh -- k x k box downsampling of the resident image pair (sid_downsample_pair).
//
// Output pixel (i, j) of each image: 0 if any of the k*k source pixels of rows k*i ... k*i+k-1, columns
// k*j ... k*j+k-1 is 0 (invalid), else floor(mean + 0.5) in integers, (2*sum + k*k) / (2*k*k).  Integer-only, so the
// result is defined to the byte.  Bandwidth-bound: every source byte is read once with 16-byte loads.
//
// A CTA makes ds_tile_out(K) output pixels of ds_rows(K) consecutive output rows: ds_tile_out(K) is a multiple of 16,
// so the tile's first source column K*j0 is 16-byte aligned (the pitch is a multiple of 16 and the base 256-byte
// aligned).  Thread t first issues the loads of chunk t (16 source columns) of all ds_rows(K) * K source rows -- 8 or
// more loads in flight per thread -- and sums each output row's K source rows as two 16-bit lanes per 32-bit word (at
// most 16 * 255 = 4080 per lane) with a byte mask of zeros.  Then, one output row at a time, it leaves its 16 column
// sums in shared memory, each with its zero flag at bit 20, and every thread adds K column sums per output pixel: at
// most 16 * 4080 < 2^20 without a flag, and at least one flag makes the total >= 2^20.  Byte b of chunk t sits at
// col[b * DS_COL_STRIDE + t]: the stores are conflict-free and the odd stride spreads the reads of neighbouring output
// pixels over the banks.  The division by 2*K*K is by a compile-time constant.  Reads stay inside the rows used and the
// 16-byte chunks that hold the columns used, which end within the pitch (>= round_up(cols, 16) + 16).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sid {

constexpr int DS_THREADS = 256;                           // 16-byte chunks per CTA and row: 4096 source columns at most
constexpr int DS_COL_STRIDE = DS_THREADS + 1;
__host__ __device__ constexpr int ds_tile_out(int k) { return (DS_THREADS * 16 / k) / 16 * 16; }
__host__ __device__ constexpr int ds_rows(int k) { return k >= 8 ? 1 : 8 / k; }   // output rows per CTA

struct DsImage {
    const uint8_t *src;
    long long src_pitch;
    uint8_t *dst;
    long long dst_pitch;
    int rows_out, cols_out;
};

// grid = (ceil(max rows_out / ds_rows(K)), ceil(max cols_out / ds_tile_out(K)), 2): blockIdx.z selects the image.
template <int K>
__global__ void __launch_bounds__(DS_THREADS) downsample_kernel(DsImage im1, DsImage im2) {
    constexpr int R = ds_rows(K), TILE = ds_tile_out(K);
    __shared__ uint32_t col[16 * DS_COL_STRIDE];
    const DsImage im = blockIdx.z ? im2 : im1;
    const int i0 = blockIdx.x * R;
    const int j0 = blockIdx.y * TILE;
    if (i0 >= im.rows_out || j0 >= im.cols_out) return;               // whole CTA: no barrier is skipped by part of it
    const int n_rows = min(R, im.rows_out - i0);
    const int n_out = min(TILE, im.cols_out - j0);
    const int t = threadIdx.x;
    const bool loads = t < ((K * n_out + 15) >> 4);
    const uint8_t *p = im.src + (long long)K * i0 * im.src_pitch + (long long)K * j0 + 16 * t;
    uint4 v[R * K];
#pragma unroll
    for (int y = 0; y < R * K; ++y)
        v[y] = (loads && y < n_rows * K) ? __ldg(reinterpret_cast<const uint4 *>(p + (long long)y * im.src_pitch))
                                         : make_uint4(0, 0, 0, 0);
    uint8_t *dst = im.dst + (long long)i0 * im.dst_pitch + j0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (r >= n_rows) break;                                       // uniform over the CTA
        uint32_t lo[4] = {0, 0, 0, 0}, hi[4] = {0, 0, 0, 0}, zero[4] = {0, 0, 0, 0};
#pragma unroll
        for (int y = 0; y < K; ++y) {
            const uint32_t w[4] = {v[r * K + y].x, v[r * K + y].y, v[r * K + y].z, v[r * K + y].w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                lo[q] += w[q] & 0x00ff00ffu;                          // bytes 0, 2
                hi[q] += (w[q] >> 8) & 0x00ff00ffu;                   // bytes 1, 3
                zero[q] |= __vcmpeq4(w[q], 0u);
            }
        }
        if (r) __syncthreads();                                       // the previous row's sums have been read
        uint32_t *c = col + t;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            c[(4 * q + 0) * DS_COL_STRIDE] = (lo[q] & 0xffffu) | ((zero[q] & 0x000000ffu) ? (1u << 20) : 0u);
            c[(4 * q + 1) * DS_COL_STRIDE] = (hi[q] & 0xffffu) | ((zero[q] & 0x0000ff00u) ? (1u << 20) : 0u);
            c[(4 * q + 2) * DS_COL_STRIDE] = (lo[q] >> 16) | ((zero[q] & 0x00ff0000u) ? (1u << 20) : 0u);
            c[(4 * q + 3) * DS_COL_STRIDE] = (hi[q] >> 16) | ((zero[q] & 0xff000000u) ? (1u << 20) : 0u);
        }
        __syncthreads();
        for (int j = t; j < n_out; j += DS_THREADS) {
            uint32_t s = 0;
#pragma unroll
            for (int x = 0; x < K; ++x) s += col[((K * j + x) & 15) * DS_COL_STRIDE + ((K * j + x) >> 4)];
            dst[j] = s >= (1u << 20) ? (uint8_t)0 : (uint8_t)((2u * s + (uint32_t)(K * K)) / (uint32_t)(2 * K * K));
        }
        dst += im.dst_pitch;
    }
}

}  // namespace sid
