// CMA-ES rank-mu covariance term on the tensor cores:  dC = sum_k w_k y_k y_k^T = Y^T diag(w) Y   (the arithmetic inside
// es.tell, cma_es.py:90; Hansen tutorial arXiv:1604.00772 eq. 47) as a symmetric rank-k update with split-fp16 operands.
//
//   Z  = diag(sqrt|w|) Y S         (so that dC = S^-1 (Zs^T Z) S^-1 with Zs = diag(sign w) Z)
//   S  = diag(2^e_j)               per-coordinate power of two: max_k |Z_kj| lands in [2^14, 2^15).  Coordinate j of y has
//                                  scale sqrt(C_jj), which CMA-ES learns and which spreads over many decades on ill-conditioned
//                                  problems; unscaled, small coordinates lose lo to fp16 subnormals and large ones overflow hi
//   exponents  Y [lambda][n] fp32 -> e [n] int32 (one coalesced read of Y)
//   pre-pass   Y [lambda][n] fp32 -> Zs_hi, Zs_lo, Z_hi, Z_lo  [n][lambda_pad] fp16, k contiguous (K-major), x = hi + lo
//   main       per 128 x 256 output tile touching the upper triangle:  D += A_hi B_hi^T + A_lo B_hi^T + A_hi B_lo^T
//              (tcgen05.mma kind::f16, fp32 accumulation in TMEM; the dropped lo*lo term is 2^-22 relative), operand
//              tiles brought in by TMA (cp.async.bulk.tensor.2d, SWIZZLE_128B) through a two-stage mbarrier pipeline:
//              warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM allocation), warps 2-5 = epilogue (tcgen05.ld, times
//              2^-e_i then 2^-e_j: both exact, -> global)
//   output     the full symmetric matrix (upper entry written to both sides: exactly symmetric), or the packed
//              upper-triangular tiles of des_cma_rank_mu_packed (the payload of the cross-rank sum)
//
// The fp32 FFMA kernel of des_cma.cu (36 % of the CUDA-core peak in round 1) stays as the small-n / no-workspace path.
// Accuracy: measured against the fp64 restatement in tests/test_gpu_cma.py at the same 1e-5 (both norms) bar, and entry by
// entry (|err_ij| <= 1e-5 sqrt(A_ii A_jj), A = sum_k |w_k| y_k y_k^T) over operand scales in tests/test_gpu_cma_range.py.
#include <cuda.h>
#include <stddef.h>
#include "des_common.cuh"
#include "des_tc.cuh"

namespace des {
namespace cmatc {

using namespace tc;

constexpr int kBM = 128, kBN = 256, kBK = 64;
constexpr int kStages = 2;
constexpr int kABytes = kBM * kBK * 2, kBBytes = kBN * kBK * 2;
constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;             // A_hi | A_lo | B_hi | B_lo = 96 KB
constexpr int kThreads = 6 * 32;

// e_j is capped so that 2^e_j and 2^-e_j are normal floats and multiplying by them is exact; the cap only binds for
// columns whose largest |z| is below 2^-112
constexpr int kExpMax = 126;

__device__ __forceinline__ float pow2f(int e) { return __int_as_float((127 + e) << 23); }     // 2^e for -126 <= e <= 127

// ---- exponent pass: e_j such that max_k |sqrt|w_k| y_kj| * 2^e_j is in [2^14, 2^15) ------------------------------------
// (hi is at most 2^15, so finite, and lo is a normal fp16 for entries within about 2^-17 of the column's largest).  A column
// that is all zero, or holds an inf or NaN, gets e_j = 0: the non-finite value stays in row and column j.
__global__ void __launch_bounds__(1024) cma_exponent_kernel(int *__restrict__ exps, const float *__restrict__ Y,
                                                            const float *__restrict__ w, int64_t lambda, int64_t n) {
    __shared__ float sqrt_w[1024];
    __shared__ uint32_t part[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 32 columns x 32 slices of k
    const int64_t j = (int64_t)blockIdx.x * 32 + tx;
    // max of |z| as bit patterns: for non-negative floats their order is the order of the values, and NaN sorts above inf
    uint32_t m = 0;
    for (int64_t k0 = 0; k0 < lambda; k0 += 1024) {
        // sqrt|w_k| from shared memory: with the sqrtf (and its slow-path call) out of the loop, the loads of Y batch up
        __syncthreads();
        sqrt_w[threadIdx.x] = k0 + threadIdx.x < lambda ? sqrtf(fabsf(__ldg(w + k0 + threadIdx.x))) : 0.f;
        __syncthreads();
        const int kn = (int)min((int64_t)1024, lambda - k0);
        if (j < n) {
            const float *y = Y + k0 * n + j;
#pragma unroll 16
            for (int r = ty; r < kn; r += 32) m = max(m, __float_as_uint(fabsf(sqrt_w[r] * __ldg(y + (int64_t)r * n))));
        }
    }
    part[ty][tx] = m;
    __syncthreads();
    if (ty == 0 && j < n) {
        for (int r = 1; r < 32; ++r) m = max(m, part[r][tx]);
        int e = 0;
        if (m != 0u && m < 0x7f800000u) {
            const int lg = m >= 0x00800000u ? (int)(m >> 23) - 127 : -118 - __clz((int)m);   // floor(log2 max), subnormals too
            e = min(14 - lg, kExpMax);
        }
        exps[j] = e;
    }
}

// ---- pre-pass: transpose + scale + split --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cma_split_kernel(__half *__restrict__ zs_hi, __half *__restrict__ zs_lo,
                                                        __half *__restrict__ z_hi, __half *__restrict__ z_lo,
                                                        const float *__restrict__ Y, const float *__restrict__ w,
                                                        const int *__restrict__ exps, int64_t lambda, int64_t lambda_pad,
                                                        int64_t n) {
    __shared__ float tile[32][33];
    __shared__ float sgn[32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 32 x 8
    const int64_t k0 = (int64_t)blockIdx.y * 32, j0 = (int64_t)blockIdx.x * 32;
    const float scale = j0 + tx < n ? pow2f(__ldg(exps + j0 + tx)) : 1.f;
    for (int r = ty; r < 32; r += 8) {
        const int64_t k = k0 + r, j = j0 + tx;
        float v = 0.f;
        if (k < lambda && j < n) v = (sqrtf(fabsf(__ldg(w + k))) * __ldg(Y + k * n + j)) * scale;   // same z as the exponent pass
        tile[r][tx] = v;
    }
    if (threadIdx.x < 32) sgn[threadIdx.x] = (k0 + threadIdx.x < lambda && __ldg(w + k0 + threadIdx.x) < 0.f) ? -1.f : 1.f;
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {                               // row j0 + r of the outputs, k = k0 + tx
        const int64_t j = j0 + r, k = k0 + tx;
        if (j < n && k < lambda_pad) {
            const float z = tile[tx][r];
            const __half h = __float2half_rn(z);
            const __half l = __float2half_rn(z - __half2float(h));
            const int64_t o = j * lambda_pad + k;
            z_hi[o] = h;
            z_lo[o] = l;
            const float s = sgn[tx];
            zs_hi[o] = __float2half_rn(s * __half2float(h));
            zs_lo[o] = __float2half_rn(s * __half2float(l));
        }
    }
}

struct Args {
    float *out;
    const int *exps;         // e_j of the exponent pass
    int64_t n;
    int k_stages;            // lambda_pad / 64
    int tiles_m, tiles_n;    // 128-row and 256-column blocks
    int packed, ptile, ptiles_per_side;
};

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

// one lane of a fully converged warp: the loop around it runs on the whole warp so that every operand of the TMA / MMA
// instructions is warp-uniform (inside `if (lane == 0)` ptxas wraps each of them in an ELECT / R2UR.BROADCAST loop)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

struct Bars {
    uint64_t full[kStages], empty[kStages], acc_full;
    uint32_t tmem_base;
    float unscale_col[kBN];  // 2^-e_j of the tile's columns
};

__global__ void __launch_bounds__(kThreads, 1) cma_syrk_kernel(Args a, const __grid_constant__ CUtensorMap map_a_hi,
                                                               const __grid_constant__ CUtensorMap map_a_lo,
                                                               const __grid_constant__ CUtensorMap map_b_hi,
                                                               const __grid_constant__ CUtensorMap map_b_lo) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    Bars *bars = reinterpret_cast<Bars *>(smem + kStages * kStageBytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // tile (bi, bj): 128-row block bi, 256-column block bj >= bi / 2 (the blocks that touch the upper triangle)
    int bi = 0, rem = blockIdx.x;
    while (rem >= a.tiles_n - (bi >> 1)) { rem -= a.tiles_n - (bi >> 1); ++bi; }
    const int bj = (bi >> 1) + rem;
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < kStages; ++s) {
                mbar_init(smem_u32(&bars->full[s]), 1);
                mbar_init(smem_u32(&bars->empty[s]), 1);
            }
            mbar_init(smem_u32(&bars->acc_full), 1);
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc(smem_u32(&bars->tmem_base), 512);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars->tmem_base;

    const uint32_t smem_addr = smem_u32(smem), bars_addr = smem_u32(bars);
    if (warp == 0) {
        // ---- TMA producer (whole warp converged, one elected lane issues)
        for (int ks = 0; ks < a.k_stages; ++ks) {
            const int s = ks % kStages, use = ks / kStages;
            if (use > 0) mbar_wait(bars_addr + (uint32_t)offsetof(Bars, empty) + 8u * s, (use - 1) & 1);
            const uint32_t bar = bars_addr + (uint32_t)offsetof(Bars, full) + 8u * s;
            const uint32_t base = smem_addr + (uint32_t)(s * kStageBytes);
            if (elect_one()) {
                mbar_expect_tx(bar, kStageBytes);
                tma_load_2d(base, &map_a_hi, ks * kBK, bi * kBM, bar);
                tma_load_2d(base + kABytes, &map_a_lo, ks * kBK, bi * kBM, bar);
                tma_load_2d(base + 2 * kABytes, &map_b_hi, ks * kBK, bj * kBN, bar);
                tma_load_2d(base + 2 * kABytes + kBBytes, &map_b_lo, ks * kBK, bj * kBN, bar);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ---- MMA issuer (whole warp converged, one elected lane issues)
        constexpr uint32_t idesc = idesc_f16(kBM, kBN);
        const uint32_t tm = __shfl_sync(0xffffffffu, tmem, 0);
        for (int ks = 0; ks < a.k_stages; ++ks) {
            const int s = ks % kStages, use = ks / kStages;
            mbar_wait(bars_addr + (uint32_t)offsetof(Bars, full) + 8u * s, use & 1);
            tc_fence_after();
            const uint32_t base = smem_addr + (uint32_t)(s * kStageBytes);
            if (elect_one()) {
#pragma unroll
                for (int k = 0; k < kBK / 16; ++k) {
                    const uint64_t ah = smem_desc_sw128(base) + (uint64_t)(k * 2);
                    const uint64_t al = smem_desc_sw128(base + kABytes) + (uint64_t)(k * 2);
                    const uint64_t bh = smem_desc_sw128(base + 2 * kABytes) + (uint64_t)(k * 2);
                    const uint64_t bl = smem_desc_sw128(base + 2 * kABytes + kBBytes) + (uint64_t)(k * 2);
                    // two accumulators, one per half of K, added with round-to-nearest in the epilogue: the tensor cores
                    // truncate when they align the fp32 accumulator, which biases long sums of same-sign terms (the
                    // diagonal: -7e-6 relative at K = 1024 with one accumulator)
                    const int half = ks >= (a.k_stages + 1) / 2 ? 1 : 0;
                    const bool first = (k == 0) && (ks == 0 || ks == (a.k_stages + 1) / 2);
                    const uint32_t d = tm + (uint32_t)(half * kBN);
                    mma_ss(d, ah, bh, idesc, !first);
                    mma_ss(d, al, bh, idesc, 1);
                    mma_ss(d, ah, bl, idesc, 1);
                }
                mma_commit(bars_addr + (uint32_t)offsetof(Bars, empty) + 8u * s);
                if (ks == a.k_stages - 1) mma_commit(bars_addr + (uint32_t)offsetof(Bars, acc_full));
            }
            __syncwarp();
        }
    } else {
        // ---- epilogue: TMEM lane quadrant = warp id % 4; lane = output row
        const int q = warp & 3;
        const int64_t i = (int64_t)bi * kBM + q * 32 + lane;
        const int64_t n = a.n;
        // the unscaling factors of the tile's rows and columns are read while the MMAs run (padding beyond n: factor 1)
        const float unscale_i = i < n ? pow2f(-__ldg(a.exps + i)) : 1.f;
        for (int c = threadIdx.x - 64; c < kBN; c += kThreads - 64) {
            const int64_t j = (int64_t)bj * kBN + c;
            bars->unscale_col[c] = j < n ? pow2f(-__ldg(a.exps + j)) : 1.f;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kThreads - 64) : "memory");     // the four epilogue warps
        mbar_wait(smem_u32(&bars->acc_full), 0);
        tc_fence_after();
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16);
        // packed tiles are padded to a multiple of their side: the padding must be written too (zeros from the TMA fill)
        const int64_t jlimit = a.packed ? (int64_t)a.ptiles_per_side * a.ptile : n;
        for (int c0 = 0; c0 < kBN; c0 += 32) {
            const int64_t j0 = (int64_t)bj * kBN + c0;
            if (j0 >= jlimit) break;                                  // warp-uniform
            if (!a.packed && j0 + 31 < (int64_t)bi * kBM + q * 32) continue;   // whole chunk below the diagonal for every lane
            uint32_t v[32];
            tmem_ld32(taddr + (uint32_t)c0, v);
            tmem_wait_ld();
            if (a.k_stages > 1) {                                     // second half of K (its own accumulator)
                uint32_t v2[32];
                tmem_ld32(taddr + (uint32_t)(kBN + c0), v2);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) + __uint_as_float(v2[e]));
            }
            // undo S on both sides: two separate power-of-two multiplies, each exact (one factor 2^-(e_i + e_j) may not
            // be a float)
#pragma unroll
            for (int e = 0; e < 32; ++e)
                v[e] = __float_as_uint((__uint_as_float(v[e]) * unscale_i) * bars->unscale_col[c0 + e]);
            if (a.packed) {
                // packed upper tiles of side ptile: element (i, j) lives in tile (i / ptile, j / ptile), bi' <= bj'
                const int64_t pb_i = i / a.ptile, pb_j = j0 / a.ptile;
                if (i < (int64_t)a.ptiles_per_side * a.ptile && pb_i <= pb_j) {
                    const int64_t t = pb_i * a.ptiles_per_side - pb_i * (pb_i - 1) / 2 + (pb_j - pb_i);
                    float4 *dst = reinterpret_cast<float4 *>(a.out + t * a.ptile * a.ptile + (i % a.ptile) * a.ptile + (j0 % a.ptile));
#pragma unroll
                    for (int e = 0; e < 8; ++e)
                        dst[e] = make_float4(__uint_as_float(v[4 * e]), __uint_as_float(v[4 * e + 1]),
                                             __uint_as_float(v[4 * e + 2]), __uint_as_float(v[4 * e + 3]));
                }
            } else {
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const int64_t j = j0 + e;
                    const float x = __uint_as_float(v[e]);
                    if (i < n && j < n && j >= i) {
                        a.out[i * n + j] = x;
                        if (j > i) a.out[j * n + i] = x;                // mirrored: exactly symmetric
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 512);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
        else
            cudaGetLastError();
    }
    return fn;
}

static int64_t lambda_pad_of(int64_t lambda) { return (lambda + kBK - 1) / kBK * kBK; }

}  // namespace cmatc
}  // namespace des

extern "C" DES_API size_t des_cma_tc_workspace_bytes(int64_t n, int64_t lambda_local) {
    if (n <= 0 || lambda_local <= 0) return 0;
    // Zs_hi | Zs_lo | Z_hi | Z_lo | e, after aligning the base to 1024 B
    return 4 * (size_t)n * (size_t)des::cmatc::lambda_pad_of(lambda_local) * sizeof(__half) + (size_t)n * sizeof(int) + 1024;
}

extern "C" DES_API int des_cma_rank_mu_tc(float *out_dev, const float *Y_dev, const float *w_dev, int64_t lambda_local, int64_t n,
                                          int packed, void *workspace_dev, size_t workspace_bytes, void *stream) {
    using namespace des;
    using namespace des::cmatc;
    DES_REQUIRE(n > 0 && lambda_local > 0, "des_cma_rank_mu_tc: bad sizes lambda=%lld n=%lld", (long long)lambda_local, (long long)n);
    DES_REQUIRE(n < ((int64_t)1 << 20), "des_cma_rank_mu_tc: n too large");
    DES_REQUIRE(out_dev && Y_dev && w_dev, "des_cma_rank_mu_tc: NULL pointer");
    const size_t need = des_cma_tc_workspace_bytes(n, lambda_local);
    if (!workspace_dev || workspace_bytes < need) {
        set_error("des_cma_rank_mu_tc: workspace %zu B < required %zu B", workspace_bytes, need);
        return DES_ERR_WORKSPACE;
    }
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) {
        set_error("des_cma_rank_mu_tc: cuTensorMapEncodeTiled is not available from this driver");
        return DES_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t lp = lambda_pad_of(lambda_local);
    __half *base = reinterpret_cast<__half *>(((uintptr_t)workspace_dev + 1023) & ~(uintptr_t)1023);
    __half *zs_hi = base, *zs_lo = base + n * lp, *z_hi = base + 2 * n * lp, *z_lo = base + 3 * n * lp;
    int *exps = reinterpret_cast<int *>(base + 4 * n * lp);
    cma_exponent_kernel<<<(unsigned)((n + 31) / 32), 1024, 0, st>>>(exps, Y_dev, w_dev, lambda_local, n);
    DES_LAUNCH_CHECK("cma_exponent_kernel");
    cma_split_kernel<<<dim3((unsigned)((n + 31) / 32), (unsigned)(lp / 32)), 256, 0, st>>>(zs_hi, zs_lo, z_hi, z_lo, Y_dev, w_dev,
                                                                                          exps, lambda_local, lp, n);
    DES_LAUNCH_CHECK("cma_split_kernel");
    CUtensorMap maps[4];
    __half *ptrs[4] = {zs_hi, zs_lo, z_hi, z_lo};
    for (int m = 0; m < 4; ++m) {
        const cuuint64_t gdim[2] = {(cuuint64_t)lp, (cuuint64_t)n};
        const cuuint64_t gstride[1] = {(cuuint64_t)lp * sizeof(__half)};
        const cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)(m < 2 ? kBM : kBN)};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult cr = enc(&maps[m], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, ptrs[m], gdim, gstride, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr != CUDA_SUCCESS) {
            set_error("des_cma_rank_mu_tc: cuTensorMapEncodeTiled failed (%d)", (int)cr);
            return DES_ERR_CUDA;
        }
    }
    Args a;
    a.out = out_dev; a.exps = exps; a.n = n; a.k_stages = (int)(lp / kBK);
    a.tiles_m = (int)((n + kBM - 1) / kBM); a.tiles_n = (int)((n + kBN - 1) / kBN);
    a.packed = packed ? 1 : 0;
    a.ptile = n <= 2048 ? 64 : 128;
    a.ptiles_per_side = (int)((n + a.ptile - 1) / a.ptile);
    int64_t tiles = 0;
    for (int bi = 0; bi < a.tiles_m; ++bi) tiles += a.tiles_n - (bi >> 1);
    const size_t smem = 1024 + (size_t)kStages * kStageBytes + sizeof(Bars);
    DES_CUDA(cudaFuncSetAttribute(cma_syrk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cma_syrk_kernel<<<(unsigned)tiles, kThreads, smem, st>>>(a, maps[0], maps[1], maps[2], maps[3]);
    DES_LAUNCH_CHECK("cma_syrk_kernel");
    return DES_OK;
}
