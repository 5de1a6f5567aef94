// LoRA merge into packed weights (sdk_lora_merge, include/sdb200.h):
//
//   dst[row_off + row_step*n][k] = cast( base[n][k] + sum_j up[n][j] * down[j][k] )      n < N, k < K
//
// One CTA owns a 64-row x 64-column output tile -- exactly one k-block row run of the k-block-major layout [K/64][rows][64] --
// stages r in chunks of RC through shared memory (up transposed, so a warp reads one broadcast row and 16 consecutive
// columns) and keeps a 4x4 register block per thread.  Plain fp32 FFMA with fp32 factors, j in increasing order: no tensor core,
// so the result is the same on every launch shape and r = 0 reproduces the packer's cast bit for bit (bf16: round to nearest even,
// as torch's .to(torch.bfloat16)).
//
// Launched WITHOUT programmatic dependent launch: the tensor-core GEMMs fetch their first weight tiles before griddepcontrol.wait
// because packed weights are stream constants (SdkTcGemmDesc.w_const).  The merge writes them, so the next launch after it must
// not start before the merge has completed; every program also begins with a non-PDL kernel, which keeps that true.
#define SDK_PDL_CAT 8
#include "common.cuh"
#include "../../include/sdb200.h"

namespace {

constexpr int TILE = 64;
constexpr int RC = 32;           // rank chunk staged per pass
constexpr int THREADS = 256;     // 16 x 16 threads, 4 x 4 outputs each

template <typename T, int LAYOUT>
__global__ void __launch_bounds__(THREADS) lora_merge_kernel(const float* __restrict__ base, int64_t ld_base,
                                                             const float* __restrict__ up, const float* __restrict__ down, int r,
                                                             T* __restrict__ dst, int dst_rows, int row_off, int row_step,
                                                             int N, int K) {
    __shared__ float s_up[RC][TILE + 1];   // [j][row], padded: the transposing store is conflict-free
    __shared__ float s_dn[RC][TILE];       // [j][col]
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int n0 = blockIdx.y * TILE, k0 = blockIdx.x * TILE;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[i][c] = -0.0f;         // x + -0 == x for every x, -0 included: r = 0 is a plain copy
    for (int j0 = 0; j0 < r; j0 += RC) {
        for (int e = threadIdx.x; e < RC * TILE; e += THREADS) {
            const int j = e / TILE, x = e % TILE;               // x: column of the tile (down) / row of the tile (up)
            const int jj = j0 + j;
            s_dn[j][x] = (jj < r && k0 + x < K) ? down[(int64_t)jj * K + k0 + x] : 0.0f;
            const int uj = e % RC, un = e / RC;                  // up[n][j]: consecutive threads on consecutive j
            s_up[uj][un] = (j0 + uj < r && n0 + un < N) ? up[(int64_t)(n0 + un) * r + j0 + uj] : 0.0f;
        }
        __syncthreads();
        const int jn = min(RC, r - j0);
        for (int j = 0; j < jn; ++j) {
            float u[4], d[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = s_up[j][ty + 16 * i];
#pragma unroll
            for (int c = 0; c < 4; ++c) d[c] = s_dn[j][tx + 16 * c];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[i][c] = fmaf(u[i], d[c], acc[i][c]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty + 16 * i;
        if (n >= N) continue;
        const int64_t drow = (int64_t)row_off + (int64_t)row_step * n;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int k = k0 + tx + 16 * c;
            if (k >= K) continue;
            const float v = base[(int64_t)n * ld_base + k] + acc[i][c];
            const int64_t o = LAYOUT == 0 ? drow * K + k : ((int64_t)(k / TILE) * dst_rows + drow) * TILE + (k % TILE);
            dst[o] = from_f32<T>(v);
        }
    }
}

template <typename T, int LAYOUT>
cudaError_t launch(const float* base, int64_t ld_base, const float* up, const float* down, int r, void* dst, int dst_rows,
                   int row_off, int row_step, int N, int K, cudaStream_t s) {
    const dim3 grid((K + TILE - 1) / TILE, (N + TILE - 1) / TILE);
    lora_merge_kernel<T, LAYOUT><<<grid, THREADS, 0, s>>>(base, ld_base, up, down, r, static_cast<T*>(dst), dst_rows, row_off,
                                                          row_step, N, K);
    return cudaPeekAtLastError();
}

}  // namespace

extern "C" int sdk_lora_merge(const float* base, int64_t ld_base, const float* up, const float* down, int r, void* dst,
                              int dst_dtype, int dst_layout, int dst_rows, int row_off, int row_step, int N, int K, void* stream) {
    SDK_CHECK_ARG(base && dst, "sdk_lora_merge: base and dst must be non-NULL");
    SDK_CHECK_ARG(N > 0 && K > 0 && ld_base >= K, "sdk_lora_merge: bad sizes N=%d K=%d ld_base=%lld", N, K, (long long)ld_base);
    SDK_CHECK_ARG(r >= 0 && (r == 0 || (up && down)), "sdk_lora_merge: r=%d needs up and down factors", r);
    SDK_CHECK_ARG(dst_dtype == SDK_F32 || dst_dtype == SDK_BF16, "sdk_lora_merge: bad dst dtype %d", dst_dtype);
    SDK_CHECK_ARG(dst_layout == SDK_LORA_ROW_MAJOR || (dst_layout == SDK_LORA_KBLOCK_MAJOR && K % 64 == 0),
                  "sdk_lora_merge: bad layout %d for K=%d", dst_layout, K);
    SDK_CHECK_ARG(row_off >= 0 && row_step >= 1 && (int64_t)row_off + (int64_t)row_step * (N - 1) < (int64_t)dst_rows,
                  "sdk_lora_merge: rows %d + %d*(N-1) outside dst_rows=%d", row_off, row_step, dst_rows);
    const cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e;
    if (dst_dtype == SDK_F32)
        e = dst_layout == SDK_LORA_ROW_MAJOR ? launch<float, 0>(base, ld_base, up, down, r, dst, dst_rows, row_off, row_step, N, K, s)
                                             : launch<float, 1>(base, ld_base, up, down, r, dst, dst_rows, row_off, row_step, N, K, s);
    else
        e = dst_layout == SDK_LORA_ROW_MAJOR
                ? launch<__nv_bfloat16, 0>(base, ld_base, up, down, r, dst, dst_rows, row_off, row_step, N, K, s)
                : launch<__nv_bfloat16, 1>(base, ld_base, up, down, r, dst, dst_rows, row_off, row_step, N, K, s);
    if (e != cudaSuccess) return sdk_fail(SDK_ERR_CUDA, "sdk_lora_merge: launch failed: %s", cudaGetErrorString(e));
    return SDK_OK;
}
