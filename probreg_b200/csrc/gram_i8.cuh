// gram_i8.cuh -- the Gram-matrix product  out[c][i] = sum_j G_ij X[c][j],  G_ij = 2^-(|a_i - a_j|^2),  with EXACT accumulation on the
// 5th-generation tensor cores: both operands are cut into 8-bit digits and multiplied with tcgen05.mma kind::i8 (unsigned x signed,
// 32-bit integer accumulators in TMEM).  These are the products of the low-rank range finder (probreg/cpd.py:296-297 with
// G = rbf_kernel(Y, Y, beta) of transformation.py:91-102, never stored); the CUDA-core kernel lr_gram_apply_kernel (lowrank.cuh) is
// the reference they are checked against.  Integer MMAs do not round -- an FP32 TMEM accumulation truncates once per MMA (measured:
// a systematic shrink of ~1e-5 over a 2048-point chunk, DESIGN 4c) -- so the only errors are the two quantisations (2^-24 absolute
// on G, 2^-23 of the column maximum on X), at the level of the float32 G the reference itself uses (cc/math_utils.cc:17-19).
//
// Fixed point ("Ozaki splitting" with integer digits):
//     g_ij = round(2^23 G_ij) in [0, 2^23]         = a0 2^16 + a1 2^8 + a2,     a_s in [0, 255]        (unsigned digits, a0 <= 128)
//     x_cj = round(2^22 X[c][j] / max_j |X[c][j]|) = b0 2^16 + b1 2^8 + b2,     b_t in [-128, 127]     (balanced digits, |b0| <= 64)
//     g x  = sum_{s,t} a_s b_t 2^(8 (4 - s - t)):   the products of level l = s + t share one accumulator,
//            levels 0, 1, 2 are kept (6 MMAs per 32 points), levels 3 and 4 (< 2^-22 of the largest term) are dropped.
// An accumulator receives at most 3 products of magnitude < 2^15 per point: exact in int32 for chunks of up to 16384 points.
// The epilogue joins the three levels in FP64 (exact) and applies the column scale; chunk partials are added in a fixed order.
//
// gi_gram_ts_kernel: CTA = 128 rows of G x up to 112 columns (3 accumulators x 112 columns of TMEM).  The columns of X are taken in
// passes of <= 112, one launch each, and G is regenerated per pass (the generators need ~2/3 of the MMA time).  Persistent over work
// units {row tile, j-chunk}, 32-point stages (one MMA K-step), 22 warps:
//     warp 0       producer: per stage, the B image (three digit planes of X, 12 KB) and the stage's j-points, two bulk copies
//     warp 1       TMEM allocation; walks the pipeline converged, one elected lane issues the 6 MMAs of a stage and the commits
//     warps 2-5    epilogue: tcgen05.ld the three int32 levels, join them in FP64, store the chunk partial
//     warps 6-21   generators: four threads per row of the tile, 8 points each; digits of round(2^23 G) into the TMEM A ring
// TMEM (512 columns): the accumulators in [0, 3 n16); behind column 3 GI_NMAX = 336 the A ring of GI_TS_STAGES = 7 stages x 3 digit
// planes x 8 columns (lane = row of the tile, 4 bytes per column): 504 columns.  A warp can only reach the 32 TMEM lanes of its quarter
// (warp % 4), so generator warp w owns rows 32 (w % 4) .. + 31 and points 8 ((w - 6) / 4) .. + 7 of each stage.
// mbarriers, per stage: full_a (the GI_TS_GEN generator warps have stored the A digits), full_b (the bytes of both bulk copies have
// landed), empty (tcgen05.commit after the stage's MMAs: B image and A slot free again); per work unit: acc_full (commit after the
// unit's last MMA), acc_empty (the 4 epilogue warps have drained the accumulators).
// B operand in shared memory: K-major, 32-byte rows, SWIZZLE_32B: row r at byte 32 r (8-row groups 256 B apart), the 16-byte half h
// of a row at position h ^ ((r >> 2) & 1).  The digit planes of X are stored in global memory AS the shared-memory image of each
// stage (gi_split_kernel: point block jb -> 3 planes x 4096 bytes, rows already swizzled), so a stage's B operand is ONE 12 KB bulk
// copy (cp.async.bulk, SASS UBLKCP).  A tensor-map box of 32-byte rows -- the first version of this kernel -- is limited by the TMA
// unit's row rate, measured at ~4.5 cycles per box row per SM: 336 rows = 1470 cycles per stage against 360 cycles of MMAs.
// The 1024-byte alignment the swizzle needs is declared on the extern shared array, NOT made by pointer arithmetic: that launders
// the address space and every access through the pointer becomes a generic LD/ST (profiles/r2_ncu_gi_gram_v3_source.txt).
#pragma once
#ifndef CPD_HOST_EMU
#include "kernels.cuh"

namespace cpd {

constexpr int GI_ROWS = 128;
constexpr int GI_KS = 32;              // j-points per stage = one kind::i8 MMA K-step (32 bytes per row)
constexpr int GI_NMAX = 112;           // columns per pass (3 levels x 112 = 336 TMEM columns)
constexpr int GI_PLANE = 4096;         // bytes reserved per digit plane of a stage image (n16 <= GI_NMAX rows of 32 bytes used)
constexpr int GI_PTS_BYTES = GI_KS * 16;                  // the stage's 32 j-points (float4), staged by the same TMA producer
constexpr int GI_MAX_CHUNK = 16384;

// ---- PTX wrappers -------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void gi_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// mbarrier wait.  With -DGI_DEBUG_WAIT (tools/umma_probe.cu) a wait gives up after ~1 s, records which one it was in
// gi_timeout_code and lets every later wait fall through, so a protocol error ends the kernel with a diagnosis instead of a hang.
#ifdef GI_DEBUG_WAIT
__device__ int gi_timeout_code = 0;
__device__ __forceinline__ void gi_wait(uint64_t* bar, uint32_t parity, int code) {
    const long long t0 = clock64();
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
            "selp.u32 %0, 1, 0, P1;\n"
            "}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (ok) return;
        if (*(volatile int*)&gi_timeout_code != 0) return;
        if (clock64() - t0 > 2000000000ll) { atomicCAS(&gi_timeout_code, 0, code); return; }
    }
}
#else
__device__ __forceinline__ void gi_wait(uint64_t* bar, uint32_t parity, int) { mbar_wait(bar, parity); }
#endif
// a wait that is not on the critical path (the epilogue warps wait a whole work unit for acc_full): poll with a pause, so that the
// waiting warps do not take issue slots from the generators (their spin loops were 30 % of all issued instructions)
__device__ __forceinline__ void gi_wait_relaxed(uint64_t* bar, uint32_t parity, int code) {
#ifdef GI_DEBUG_WAIT
    gi_wait(bar, parity, code);
#else
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
            "selp.u32 %0, 1, 0, P1;\n"
            "}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (ok) return;
        __nanosleep(400);
    }
#endif
}
// one lane of a converged warp (elect.sync).  The MMA-issuing warp runs its loop with all 32 lanes and elects only around the
// tcgen05 instructions: the descriptor arithmetic then stays warp-uniform and compiles to the uniform datapath.  Inside an
// `if (lane == 0)` branch the same values are per-thread registers and every tcgen05.mma needs ~8 R2UR transfers on one thread --
// the issue loop, not the tensor pipe, set the pace (tensor pipe 37 % active, profiles/r2_ncu_gi_gram_v5.txt).
__device__ __forceinline__ bool gi_elect_one() {
    uint32_t pred = 0, laneid = 0;
    asm volatile(
        "{\n"
        ".reg .b32 %%rx;\n"
        ".reg .pred %%px;\n"
        "     elect.sync %%rx|%%px, %2;\n"
        "@%%px mov.s32 %1, 1;\n"
        "     mov.s32 %0, %%rx;\n"
        "}\n"
        : "+r"(laneid), "+r"(pred)
        : "r"(0xFFFFFFFF));
    return pred != 0;
}
__device__ __forceinline__ void gi_tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void gi_tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void gi_tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void gi_tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// completion of every tcgen05.mma issued so far by this thread -> one arrival on the mbarrier (implies fence::before_thread_sync)
__device__ __forceinline__ void gi_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major, SWIZZLE_32B (layout type 6), 8-row groups 256 bytes apart
__device__ __forceinline__ uint64_t gi_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | (1ull << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46) | (6ull << 61);
}
// D = S32 (2 at [4,6)), A = unsigned 8-bit (0 at [7,10)), B = signed 8-bit (1 at [10,13)), K-major, N >> 3 at [17,23), M >> 4 at [24,29)
__host__ __device__ __forceinline__ uint32_t gi_instr_desc(int n) {
    return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ uint32_t gi_row_half_offset(int r, int h) { return (uint32_t)(r * 32 + ((h ^ ((r >> 2) & 1)) << 4)); }
__device__ __forceinline__ void gi_tmem_ld16(uint32_t taddr, int (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = (int)r[k];
}

// first-use self-check: the largest |a - b| and |b| over rows [0, rows) of `cols` columns  ->  res[0], res[1] (one CTA)
__global__ void __launch_bounds__(THREADS)
gi_compare_kernel(const double* __restrict__ a, const double* __restrict__ b, long long ld, long long i_begin, long long rows, int cols,
                  double* __restrict__ res) {
    __shared__ double sd[THREADS], sv[THREADS];
    double d = 0.0, v = 0.0;
    for (int c = 0; c < cols; ++c)
        for (long long i = threadIdx.x; i < rows; i += THREADS) {
            const double x = a[(long long)c * ld + i_begin + i], y = b[(long long)c * ld + i_begin + i];
            d = fmax(d, fabs(x - y)); v = fmax(v, fabs(y));
            if (!(x == x)) d = 1e300;                      // NaN in the tensor-core result
        }
    sd[threadIdx.x] = d; sv[threadIdx.x] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int t = 1; t < THREADS; ++t) { d = fmax(d, sd[t]); v = fmax(v, sv[t]); }
        res[0] = d; res[1] = v;
    }
}

// ---- operand preparation -----------------------------------------------------------------------------------------------------------
// colmax[c] = max_j |X[c][j]|   (one CTA per column)
__global__ void __launch_bounds__(THREADS)
gi_colmax_kernel(const double* __restrict__ X, long long m, long long ld, double* __restrict__ colmax) {
    __shared__ double sh[THREADS / 32];
    const int c = blockIdx.x;
    double v = 0.0;
    for (long long j = threadIdx.x; j < m; j += THREADS) v = fmax(v, fabs(X[(long long)c * ld + j]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < THREADS / 32; ++w) v = fmax(v, sh[w]);
        colmax[c] = v;
    }
}
// digit planes of the columns [c0, c0 + nc) as stage images: image[jb] (jb = point block of 32) = 3 planes x GI_PLANE bytes, plane p
// holds digit p of column c (row c, 32 bytes, the two 16-byte halves swizzled like the MMA reads them).  One thread = one column x
// 16 points = one 16-byte store per plane; rows c >= nc and points j >= m are zero.
__global__ void __launch_bounds__(THREADS)
gi_split_kernel(const double* __restrict__ X, long long m, long long ld, int nc, int n16, long long ldx, const double* __restrict__ colmax,
                unsigned char* __restrict__ images) {
    const long long jh = (long long)blockIdx.x * THREADS + threadIdx.x;          // 16-point group
    const int c = blockIdx.y;
    if (jh * 16 < ldx && c < n16) {
        uint32_t w[3][4] = {{0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}};
        const double mx = c < nc ? colmax[c] : 0.0;
        if (mx > 0.0) {
            const double inv = 4194304.0 / mx;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const long long j = jh * 16 + k;
                if (j < m) {
                    const int xi = (int)rint(X[(long long)c * ld + j] * inv);                 // |xi| <= 2^22
                    const int b2 = ((xi + 128) & 255) - 128;
                    const int r1 = (xi - b2) >> 8;
                    const int b1 = ((r1 + 128) & 255) - 128;
                    const int b0 = (r1 - b1) >> 8;
                    w[0][k >> 2] |= (uint32_t)(b0 & 255) << (8 * (k & 3));
                    w[1][k >> 2] |= (uint32_t)(b1 & 255) << (8 * (k & 3));
                    w[2][k >> 2] |= (uint32_t)(b2 & 255) << (8 * (k & 3));
                }
            }
        }
        unsigned char* img = images + (jh >> 1) * (3 * GI_PLANE) + gi_row_half_offset(c, (int)(jh & 1));
#pragma unroll
        for (int p = 0; p < 3; ++p) *reinterpret_cast<uint4*>(img + p * GI_PLANE) = make_uint4(w[p][0], w[p][1], w[p][2], w[p][3]);
    }
}
// out[c][i_begin + ii] = sum over the j-chunks of part[q][c][ii] (FP64, chunk order)
__global__ void __launch_bounds__(THREADS)
gi_reduce_kernel(const double* __restrict__ part, int nq, int n16, long long ldp, int nc, long long rows, long long i_begin, long long ld,
                 double* __restrict__ out) {
    const long long ii = (long long)blockIdx.x * THREADS + threadIdx.x;
    const int c = blockIdx.y;
    if (ii < rows && c < nc) {
        double s = 0.0;
        for (int q = 0; q < nq; ++q) s += part[((long long)q * n16 + c) * ldp + ii];
        out[(long long)c * ld + i_begin + ii] = s;
    }
}

// j-points as packed pairs for the generators' f32x2 arithmetic: record k (32 bytes) = {x_2k, x_2k+1, y_2k, y_2k+1}, {z_2k, z_2k+1, 0, 0}
__global__ void __launch_bounds__(THREADS)
gi_pairs_kernel(const float4* __restrict__ pts, long long npairs, float4* __restrict__ rec) {
    const long long k = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (k < npairs) {
        const float4 p = pts[2 * k], q = pts[2 * k + 1];
        rec[2 * k] = make_float4(p.x, q.x, p.y, q.y);
        rec[2 * k + 1] = make_float4(p.z, q.z, 0.0f, 0.0f);
    }
}

constexpr int GI_TS_STAGES = 7;                        // the A ring in TMEM: 7 x 24 columns behind the 336 accumulator columns
constexpr int GI_TS_GEN = 16;                          // generator warps (four threads per row of the tile)
constexpr int GI_TS_THREADS = (6 + GI_TS_GEN) * 32;
constexpr int GI_TS_STAGE_BYTES = 3 * GI_PLANE;         // shared memory per stage: the B image only
constexpr int GI_TS_SMEM = GI_TS_STAGES * (GI_TS_STAGE_BYTES + GI_PTS_BYTES) + 1024 + 256;
__device__ __forceinline__ void gi_mma_i8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n"
        "}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void gi_tmem_st2(uint32_t taddr, uint32_t w0, uint32_t w1) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(w0), "r"(w1) : "memory");
}

// ---- the product, A operand in TENSOR MEMORY (tcgen05.mma ".ts" form) ---------------------------------------------------------------
// A in TMEM rather than in shared memory: with A in shared memory the kernel was bound by the shared-memory port (generator STS + LDS
// 51 %, tensor operand reads 42 %, profiles/r2_ncu_gi_gram_final.txt); TMEM removes the 12 KB of STS and the 24 KB of A-operand reads
// per stage.
// one column pass: images = the stage images of gi_split_kernel (jpad / 32 of them); rows [i_begin, i_end) of G;
// part[q][c][ii] (FP64) = colmax[c] 2^-45 sum_{j in chunk q} g_ij x_cj
__global__ void __launch_bounds__(GI_TS_THREADS, 1)
gi_gram_ts_kernel(const unsigned char* __restrict__ images, const float4* __restrict__ pts, const float4* __restrict__ pairs, long long jpad, int chunk,
               long long i_begin,
               long long i_end, int n16, const double* __restrict__ colmax, double* __restrict__ part, long long ldp) {
    extern __shared__ __align__(1024) unsigned char gi_smem_raw[];
    unsigned char* smem = gi_smem_raw;
    unsigned char* spts = smem + GI_TS_STAGES * GI_TS_STAGE_BYTES;            // [GI_TS_STAGES][32] float4: the j-points of each stage
    uint64_t* bars = reinterpret_cast<uint64_t*>(spts + GI_TS_STAGES * GI_PTS_BYTES);
    uint64_t* full_a = bars;
    uint64_t* full_b = bars + GI_TS_STAGES;
    uint64_t* empty = bars + 2 * GI_TS_STAGES;
    uint64_t* acc_full = bars + 3 * GI_TS_STAGES;
    uint64_t* acc_empty = bars + 3 * GI_TS_STAGES + 1;
    uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 3 * GI_TS_STAGES + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long rows = i_end - i_begin;
    const int ntiles = (int)((rows + GI_ROWS - 1) / GI_ROWS);
    const int nq = (int)((jpad + chunk - 1) / chunk);
    const long long nunits = (long long)ntiles * nq;

    if (threadIdx.x == 0) {
        for (int s = 0; s < GI_TS_STAGES; ++s) { mbar_init(&full_a[s], GI_TS_GEN); mbar_init(&full_b[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, 4);
        mbar_fence_init();
    }
    if (warp == 1) gi_tmem_alloc(tmem_base_slot, 512);
    gi_tc_fence_before();
    __syncthreads();
    gi_tc_fence_after();
    const uint32_t tmem_base = *tmem_base_slot;

    if (warp == 0) {
        // ===== TMA producer: the stage image (three digit planes of X for 32 points), one bulk copy =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (long long u = blockIdx.x; u < nunits; u += gridDim.x) {
                const int q = (int)(u / ntiles);
                const long long j0 = (long long)q * chunk;
                const int nst = (int)((min((long long)chunk, jpad - j0)) / GI_KS);
                const unsigned char* src = images + (j0 / GI_KS) * (3 * GI_PLANE);
                for (int kb = 0; kb < nst; ++kb) {
                    gi_wait(&empty[stage], phase ^ 1, 11);
                    mbar_expect_tx(&full_b[stage], (uint32_t)(3 * GI_PLANE + GI_PTS_BYTES));
                    tma_load_1d(smem + stage * GI_TS_STAGE_BYTES, src + (long long)kb * (3 * GI_PLANE), (uint32_t)(3 * GI_PLANE),
                                &full_b[stage]);
                    tma_load_1d(spts + stage * GI_PTS_BYTES, pairs + j0 + (long long)kb * GI_KS, (uint32_t)GI_PTS_BYTES, &full_b[stage]);
                    if (++stage == GI_TS_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: level l = s + t accumulates a_s x b_t; the whole warp walks the pipeline, one elected lane issues =====
        {
            const uint32_t idesc = gi_instr_desc(n16);
            uint32_t stage = 0, phase = 0, acc_phase = 0;
            for (long long u = blockIdx.x; u < nunits; u += gridDim.x) {
                const int q = (int)(u / ntiles);
                const long long j0 = (long long)q * chunk;
                const int nst = (int)((min((long long)chunk, jpad - j0)) / GI_KS);
                gi_wait(acc_empty, acc_phase ^ 1, 12);
                gi_tc_fence_after();
                for (int kb = 0; kb < nst; ++kb) {
                    gi_wait(&full_a[stage], phase, 13);
                    gi_wait(&full_b[stage], phase, 14);
                    gi_tc_fence_after();
                    const uint32_t sb = smem_u32(smem) + stage * GI_TS_STAGE_BYTES;
                    const uint32_t ta = tmem_base + (uint32_t)(3 * GI_NMAX + stage * 24);       // this stage's three A planes (8 columns each)
                    const uint32_t first = kb != 0 ? 1u : 0u;
                    if (gi_elect_one()) {
                        uint64_t b[3];
#pragma unroll
                        for (int p = 0; p < 3; ++p) b[p] = gi_smem_desc(sb + p * GI_PLANE);
                        gi_mma_i8_ts(tmem_base, ta, b[0], idesc, first);
                        gi_mma_i8_ts(tmem_base + (uint32_t)n16, ta, b[1], idesc, first);
                        gi_mma_i8_ts(tmem_base + (uint32_t)n16, ta + 8, b[0], idesc, 1u);
                        gi_mma_i8_ts(tmem_base + (uint32_t)(2 * n16), ta, b[2], idesc, first);
                        gi_mma_i8_ts(tmem_base + (uint32_t)(2 * n16), ta + 8, b[1], idesc, 1u);
                        gi_mma_i8_ts(tmem_base + (uint32_t)(2 * n16), ta + 16, b[0], idesc, 1u);
                        gi_commit(&empty[stage]);
                        if (kb == nst - 1) gi_commit(acc_full);
                    }
                    __syncwarp();
                    if (++stage == GI_TS_STAGES) { stage = 0; phase ^= 1; }
                }
                acc_phase ^= 1;
            }
        }
    } else if (warp < 6) {
        // ===== epilogue: join the three levels in FP64 (exact), scale, store the chunk partial =====
        const int quarter = warp & 3;
        uint32_t acc_phase = 0;
        for (long long u = blockIdx.x; u < nunits; u += gridDim.x) {
            const int q = (int)(u / ntiles), t = (int)(u % ntiles);
            gi_wait_relaxed(acc_full, acc_phase, 15);
            gi_tc_fence_after();
            const long long ii = (long long)t * GI_ROWS + quarter * 32 + lane;
            double* dst = part + (long long)q * n16 * ldp + ii;
            const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16);
#pragma unroll 1
            for (int c0 = 0; c0 < n16; c0 += 16) {
                int v0[16], v1[16], v2[16];
                gi_tmem_ld16(tlane + (uint32_t)c0, v0);
                gi_tmem_ld16(tlane + (uint32_t)(n16 + c0), v1);
                gi_tmem_ld16(tlane + (uint32_t)(2 * n16 + c0), v2);
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const double s = (double)v0[k] * 65536.0 + (double)v1[k] * 256.0 + (double)v2[k];      // exact: < 2^48
                    dst[(long long)(c0 + k) * ldp] = s * (colmax[c0 + k] * (1.0 / 536870912.0));           // 2^16 2^-45
                }
            }
            gi_tc_fence_before();
            __syncwarp();
            if (lane == 0) gi_mbar_arrive(acc_empty);
            acc_phase ^= 1;
        }
    } else {
        // ===== generators: FOUR threads per row (8 points each), 16 warps: four per scheduler instead of two -- the 8-warp version
        // issued at half the peak rate with every pipe below 45 % (latency, not throughput).  Digits of round(2^23 G) -> TMEM =====
        const int quarter = warp & 3, r = quarter * 32 + lane, part = (warp - 6) >> 2;          // part: which 8 of the stage's 32 points
        uint32_t stage = 0, phase = 0;
        for (long long u = blockIdx.x; u < nunits; u += gridDim.x) {
            const int q = (int)(u / ntiles), t = (int)(u % ntiles);
            const long long j0 = (long long)q * chunk;
            const int nst = (int)((min((long long)chunk, jpad - j0)) / GI_KS);
            long long i = i_begin + (long long)t * GI_ROWS + r;
            if (i >= i_end) i = i_end - 1;
            const float4 a = pts[i];
            const u64 ax2 = pack2(a.x, a.x), ay2 = pack2(a.y, a.y), az2 = pack2(a.z, a.z), magic2 = pack2(8388608.0f, 8388608.0f);
            for (int kb = 0; kb < nst; ++kb) {
                gi_wait(&full_b[stage], phase, 19);                // the j-points arrive with the B image
                const ulonglong2* bj = reinterpret_cast<const ulonglong2*>(spts + stage * GI_PTS_BYTES) + part * 8;     // 4 pair records
                // g = round(2^23 G) sits in the mantissa of 2^23 + 2^23 G (one FMA; a float -> integer conversion would go through the
                // quarter-rate XU pipe that MUFU.EX2 already loads): bytes 2, 1, 0 of the float ARE the digits a0 < 128, a1, a2.
                uint32_t gq[8];
#pragma unroll
                for (int pr = 0; pr < 4; ++pr) {
                    const ulonglong2 bxy = bj[2 * pr];
                    const u64 bz = bj[2 * pr + 1].x;
                    const u64 dx = fsub2(ax2, bxy.x), dy = fsub2(ay2, bxy.y), dz = fsub2(az2, bz);
                    const float2 uu = unpack2(ffma2(dz, dz, ffma2(dy, dy, fmul2(dx, dx))));
                    const u64 e = pack2(ex2(-uu.x), ex2(-uu.y));  // the same float32 G as the other kernels; G = 1 gives the digits (128, 0, 0)
                    const float2 tt = unpack2(ffma2(e, magic2, magic2));
                    gq[2 * pr] = __float_as_uint(tt.x);
                    gq[2 * pr + 1] = __float_as_uint(tt.y);
                }
                gi_wait(&empty[stage], phase ^ 1, 16);
                gi_tc_fence_after();                               // the MMAs that read this slot last have completed (tcgen05.commit)
                const uint32_t ta = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(3 * GI_NMAX + stage * 24 + part * 2);
#pragma unroll
                for (int p = 0; p < 3; ++p) {
                    const uint32_t sel = p == 0 ? 0x0062u : (p == 1 ? 0x0051u : 0x0040u);     // byte (2 - p) of both inputs
                    const uint32_t w0 = __byte_perm(__byte_perm(gq[0], gq[1], sel), __byte_perm(gq[2], gq[3], sel), 0x5410u);
                    const uint32_t w1 = __byte_perm(__byte_perm(gq[4], gq[5], sel), __byte_perm(gq[6], gq[7], sel), 0x5410u);
                    gi_tmem_st2(ta + (uint32_t)(p * 8), w0, w1);       // this row's 8 bytes of plane p: 2 columns
                }
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                gi_tc_fence_before();
                __syncwarp();
                if (lane == 0) gi_mbar_arrive(&full_a[stage]);
                if (++stage == GI_TS_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    }
    gi_tc_fence_before();
    __syncthreads();
    if (warp == 1) gi_tmem_dealloc(tmem_base, 512);
}

}  // namespace cpd
#endif  // CPD_HOST_EMU
