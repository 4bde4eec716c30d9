// tools/umma_probe.cu -- hardware bring-up of csrc/gram_i8.cuh (tcgen05 cannot be emulated on the CPU):
//   1. layout probe: one [128 x 32] (u8, A in tensor memory) x [32 x N] (s8) kind::i8 MMA through the kernel's descriptor / swizzle /
//      TMEM conventions against the CPU (integer results, so every entry must be equal); on a mismatch, identity patterns decode which
//      element the tensor core actually read where;
//   2. the full product G X (gi_gram_ts_kernel) against an FP64 CPU sum on sampled rows and against the CUDA-core kernel, with timings.
// Built with -DGI_DEBUG_WAIT: every mbarrier wait gives up after ~1 s and names itself, so a protocol error is reported, not a hang.
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -DGI_DEBUG_WAIT -Iprobreg_b200/csrc -Iinclude -o build/umma_probe tools/umma_probe.cu
// run:   timeout 300 build/umma_probe [points=50000] [rank=200]
#include <cuda.h>          // CUtensorMap (type only: the encode entry point is fetched from the driver at run time)
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "lowrank.cuh"
#include "gram_i8.cuh"

using namespace cpd;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at line %d: %s\n", #x, __LINE__, cudaGetErrorString(e_)); return 1; } } while (0)

static double urand(unsigned long long& s) { s = s * 6364136223846793005ull + 1442695040888963407ull; return (double)(s >> 11) / 9007199254740992.0; }

static int timeout_code() { int c = 0; cudaMemcpyFromSymbol(&c, gi_timeout_code, sizeof(int)); return c; }

// ---- layout probe: B arrives through a tensor map whose 32-byte swizzle gives the layout of gi_split_kernel's stage images ------------
__device__ __forceinline__ void gi_tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                     smem_u32(dst)),
                 "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
// four consecutive 32-bit columns of this thread's TMEM lane
__device__ __forceinline__ void gi_tmem_st4(uint32_t taddr, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(w0), "r"(w1), "r"(w2), "r"(w3) : "memory");
}

// D[128][n16] (int32) = A[128][32] (u8) x B[n16][32]^T (s8): A in tensor memory (tcgen05.st by the owning thread, ".ts" MMA)
__global__ void __launch_bounds__(128, 1)
gi_layout_probe_ts_kernel(const __grid_constant__ CUtensorMap bmap, const unsigned char* __restrict__ A, int n16, int* __restrict__ D) {
    extern __shared__ __align__(1024) unsigned char gi_smem_raw[];
    unsigned char* smem = gi_smem_raw;
    unsigned char* sb = smem;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 8192);
    uint32_t* slot = reinterpret_cast<uint32_t*>(bars + 2);
    const int warp = threadIdx.x >> 5, r = threadIdx.x;
    if (threadIdx.x == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
    if (warp == 0) gi_tmem_alloc(slot, 512);
    gi_tc_fence_before();
    __syncthreads();
    gi_tc_fence_after();
    const uint32_t tmem_base = *slot;
    if (threadIdx.x == 0) {
        mbar_expect_tx(&bars[0], (uint32_t)(n16 * 32));
        gi_tma_load_2d(sb, &bmap, 0, 0, &bars[0]);
    }
    const uint4 lo = *reinterpret_cast<const uint4*>(A + r * 32), hi = *reinterpret_cast<const uint4*>(A + r * 32 + 16);
    const uint32_t ta = tmem_base + ((uint32_t)(warp * 32) << 16) + 256u;          // A in columns 256..263
    gi_tmem_st4(ta, lo.x, lo.y, lo.z, lo.w);
    gi_tmem_st4(ta + 4, hi.x, hi.y, hi.z, hi.w);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    gi_tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) {
        gi_wait(&bars[0], 0, 27);
        gi_tc_fence_after();
        gi_mma_i8_ts(tmem_base, tmem_base + 256u, gi_smem_desc(smem_u32(sb)), gi_instr_desc(n16), 0u);
        gi_commit(&bars[1]);
    }
    gi_wait(&bars[1], 0, 28);
    gi_tc_fence_after();
    for (int c0 = 0; c0 < n16; c0 += 16) {
        int v[16];
        gi_tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
        for (int k = 0; k < 16; ++k) D[r * n16 + c0 + k] = v[k];
    }
    gi_tc_fence_before();
    __syncthreads();
    if (warp == 0) gi_tmem_dealloc(tmem_base, 512);
}

// tensor map over byte planes: [rows][ld] bytes, box {32, box_rows}, 32-byte swizzle (cuTensorMapEncodeTiled is fetched from the
// driver: no link against libcuda)
typedef CUresult (*gi_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int gi_make_map(CUtensorMap* map, const void* base, long long ld, long long rows, int box_rows) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) return -1;
    const cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld};
    const cuuint32_t box[2] = {(cuuint32_t)GI_KS, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = reinterpret_cast<gi_encode_fn>(fn)(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                                                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B,
                                                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)r;
}

// ---- kind::i8: exact integer results, so every comparison is for equality ---------------------------------------------------------
static int run_layout_i8(int n16, const std::vector<unsigned char>& A, const std::vector<signed char>& B, std::vector<int>& D) {
    unsigned char* dA; signed char* dB; int* dD;
    CK(cudaMalloc(&dA, 128 * 32)); CK(cudaMalloc(&dB, (size_t)n16 * 32)); CK(cudaMalloc(&dD, (size_t)128 * n16 * 4));
    CK(cudaMemcpy(dA, A.data(), 128 * 32, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dB, B.data(), (size_t)n16 * 32, cudaMemcpyHostToDevice));
    CK(cudaMemset(dD, 0x7f, (size_t)128 * n16 * 4));
    CUtensorMap map;
    if (gi_make_map(&map, dB, 32, n16, n16) != 0) { printf("i8 tensor map encode failed\n"); return 1; }
    CK(cudaFuncSetAttribute(gi_layout_probe_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 20000));
    gi_layout_probe_ts_kernel<<<1, 128, 20000>>>(map, dA, n16, dD);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    D.resize((size_t)128 * n16);
    CK(cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost));
    cudaFree(dA); cudaFree(dB); cudaFree(dD);
    const int tc = timeout_code();
    if (tc) { printf("i8 layout probe: wait %d timed out\n", tc); return 2; }
    return 0;
}
static int layout_tests_i8() {
    unsigned long long seed = 4242;
    int bad = 0;
    for (int n16 : {16, 112, 256}) {
        std::vector<unsigned char> A(128 * 32);
        std::vector<signed char> B((size_t)n16 * 32);
        std::vector<int> D;
        for (auto& v : A) v = (unsigned char)(urand(seed) * 256.0);
        for (auto& v : B) v = (signed char)((int)(urand(seed) * 256.0) - 128);
        const int rc = run_layout_i8(n16, A, B, D);
        if (rc) return rc;
        long long wrong = 0;
        for (int r = 0; r < 128; ++r)
            for (int n = 0; n < n16; ++n) {
                int s = 0;
                for (int k = 0; k < 32; ++k) s += (int)A[r * 32 + k] * (int)B[n * 32 + k];
                wrong += s != D[(size_t)r * n16 + n];
            }
        printf("i8 layout (A in TMEM) n=%3d: %lld of %d entries differ from the integer reference   %s\n", n16, wrong, 128 * n16, wrong ? "MISMATCH" : "OK");
        if (wrong) bad = 1;
    }
    if (bad) {
        // decode: B = identity rows (B[n][k] = (n == k), n < 32), A[r][k] = 32 (r % 8) + k: D[r][n] shows which A byte sat at (r, k = n)
        const int n16 = 32;
        std::vector<unsigned char> A(128 * 32);
        std::vector<signed char> B((size_t)n16 * 32, 0);
        std::vector<int> D;
        for (int r = 0; r < 128; ++r) for (int k = 0; k < 32; ++k) A[r * 32 + k] = (unsigned char)((r & 7) * 32 + k);
        for (int n = 0; n < 32; ++n) B[n * 32 + n] = 1;
        if (run_layout_i8(n16, A, B, D) == 0) {
            printf("decode A (identity B): D[r][n] should be 32 (r %% 8) + n; as (row %% 8, k) read:\n");
            for (int r : {0, 1, 2, 3, 4, 5, 6, 7, 8, 12, 127}) {
                printf("  r=%3d:", r);
                for (int n = 0; n < 32; ++n) printf(" (%d,%d)", D[(size_t)r * n16 + n] / 32, D[(size_t)r * n16 + n] % 32);
                printf("\n");
            }
        }
        for (int r = 0; r < 128; ++r) for (int k = 0; k < 32; ++k) A[r * 32 + k] = (r % 32 == k) ? 1 : 0;
        for (int n = 0; n < 32; ++n) for (int k = 0; k < 32; ++k) B[n * 32 + k] = (signed char)((n & 3) * 32 + k - 64);
        if (run_layout_i8(n16, A, B, D) == 0) {
            printf("decode B (identity-pattern A): D[r][n] should be 32 (n %% 4) + r %% 32 - 64; rows 0..7:\n");
            for (int r = 0; r < 8; ++r) {
                printf("  r=%3d:", r);
                for (int n = 0; n < 32; ++n) printf(" %d", D[(size_t)r * n16 + n] + 64);
                printf("\n");
            }
        }
    }
    return bad ? 3 : 0;
}

static int full_test_i8(long long m, int rank, double beta, bool time_old, int xkind) {
    const long long mpad = (m + 511) / 512 * 512;
    unsigned long long seed = 999;
    std::vector<double> Y((size_t)m * 3), X((size_t)rank * mpad, 0.0);
    for (long long i = 0; i < m; ++i) { Y[3 * i] = urand(seed); Y[3 * i + 1] = 0.6 * urand(seed); Y[3 * i + 2] = 0.3 * urand(seed); }
    for (int c = 0; c < rank; ++c)
        for (long long j = 0; j < m; ++j) {
            double v = 2.0 * urand(seed) - 1.0;
            if (xkind == 1) v *= exp(-12.0 * urand(seed)) * (1.0 + c);          // entries over 5 decades, columns of different scale
            X[(size_t)c * mpad + j] = v;
        }
    double *dY, *dX, *dOutNew, *dOutOld, *dColmax, *dPart;
    float4 *dPts, *dPairs;
    unsigned char* dPlanes;
    const long long chunk = mpad < GI_MAX_CHUNK ? mpad : GI_MAX_CHUNK;
    const int nq = (int)((mpad + chunk - 1) / chunk), ntiles = (int)((m + GI_ROWS - 1) / GI_ROWS);
    const long long ldp = (long long)ntiles * GI_ROWS;
    const int passes = (rank + GI_NMAX - 1) / GI_NMAX, per = (rank + passes - 1) / passes, n16max = (per + 15) / 16 * 16;
    CK(cudaMalloc(&dY, (size_t)m * 3 * 8)); CK(cudaMalloc(&dX, (size_t)rank * mpad * 8));
    CK(cudaMalloc(&dOutNew, (size_t)rank * mpad * 8)); CK(cudaMalloc(&dOutOld, (size_t)rank * mpad * 8));
    CK(cudaMalloc(&dPts, (size_t)mpad * 16));
    CK(cudaMalloc(&dPlanes, (size_t)(mpad / GI_KS) * 3 * GI_PLANE));
    CK(cudaMalloc(&dPairs, (size_t)mpad * 16));
    CK(cudaMalloc(&dPart, (size_t)nq * n16max * ldp * 8));
    CK(cudaMalloc(&dColmax, (size_t)(rank + 256) * 8));
    CK(cudaMemset(dColmax, 0, (size_t)(rank + 256) * 8));
    CK(cudaMemcpy(dY, Y.data(), (size_t)m * 3 * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dX, X.data(), (size_t)rank * mpad * 8, cudaMemcpyHostToDevice));
    lr_pack_kernel<<<(unsigned)((mpad + THREADS - 1) / THREADS), THREADS>>>(dY, 0.0, 0.0, 0.0, m, mpad, (float)sqrt(LOG2E / (2.0 * beta)), dPts);
    gi_pairs_kernel<<<(unsigned)((mpad / 2 + THREADS - 1) / THREADS), THREADS>>>(dPts, mpad / 2, dPairs);
    CK(cudaFuncSetAttribute(gi_gram_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GI_TS_SMEM));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float t_all = 0, t_gram = 0;
    for (int rep = 0; rep < 3; ++rep) {
        t_gram = 0;
        cudaEventRecord(e0);
        gi_colmax_kernel<<<rank, THREADS>>>(dX, m, mpad, dColmax);
        for (int c0 = 0; c0 < rank; c0 += per) {
            const int nc = per < rank - c0 ? per : rank - c0, n16 = (nc + 15) / 16 * 16;
            gi_split_kernel<<<dim3((unsigned)((mpad / 16 + THREADS - 1) / THREADS), n16), THREADS>>>(dX + (size_t)c0 * mpad, m, mpad, nc, n16, mpad, dColmax + c0, dPlanes);
            cudaEvent_t g0, g1; cudaEventCreate(&g0); cudaEventCreate(&g1);
            cudaEventRecord(g0);
            gi_gram_ts_kernel<<<sms, GI_TS_THREADS, GI_TS_SMEM>>>(dPlanes, dPts, dPairs, mpad, (int)chunk, 0, m, n16, dColmax + c0, dPart, ldp);
            cudaEventRecord(g1);
            gi_reduce_kernel<<<dim3((unsigned)((m + THREADS - 1) / THREADS), nc), THREADS>>>(dPart, nq, n16, ldp, nc, m, 0, mpad, dOutNew + (size_t)c0 * mpad);
            CK(cudaGetLastError());
            CK(cudaDeviceSynchronize());
            float tg = 0; cudaEventElapsedTime(&tg, g0, g1); t_gram += tg;
            cudaEventDestroy(g0); cudaEventDestroy(g1);
        }
        cudaEventRecord(e1);
        CK(cudaDeviceSynchronize());
        cudaEventElapsedTime(&t_all, e0, e1);
        const int tc = timeout_code();
        if (tc) { printf("i8 full kernel: wait %d timed out\n", tc); return 2; }
    }
    printf("i8 (A in TMEM): m=%lld rank=%d (%d passes of N=%d) beta=%g xkind=%d: gram kernels %.3f ms, whole product (incl. split/reduce and host syncs) %.3f ms; "
           "%.1f TFLOP/s useful\n", m, rank, passes, n16max, beta, xkind, t_gram, t_all, 2.0 * m * m * rank / (t_gram * 1e-3) / 1e12);
    float t_old = 0;
    if (time_old) {
        cudaEventRecord(e0);
        lr_gram_apply_kernel<<<dim3((unsigned)((m + THREADS - 1) / THREADS), (unsigned)((rank + LR_COLS - 1) / LR_COLS)), THREADS>>>(
            dPts, m, mpad, dX, mpad, rank, dOutOld, 0, m);
        cudaEventRecord(e1);
        CK(cudaDeviceSynchronize());
        cudaEventElapsedTime(&t_old, e0, e1);
    }
    std::vector<double> on((size_t)rank * mpad), oo((size_t)rank * mpad);
    CK(cudaMemcpy(on.data(), dOutNew, on.size() * 8, cudaMemcpyDeviceToHost));
    if (time_old) CK(cudaMemcpy(oo.data(), dOutOld, oo.size() * 8, cudaMemcpyDeviceToHost));
    std::vector<float4> P(mpad);
    CK(cudaMemcpy(P.data(), dPts, (size_t)mpad * 16, cudaMemcpyDeviceToHost));
    const int nsample = 32;
    double en = 0, eo = 0;      // per column: max |err| / max |value| of that column, then the max over columns
    std::vector<double> ref((size_t)nsample * rank), colscale(rank, 0.0);
    std::vector<long long> rowsel(nsample);
    for (int s = 0; s < nsample; ++s) {
        const long long i = (s == 0) ? 0 : (s == 1 ? m - 1 : (long long)(urand(seed) * m));
        rowsel[s] = i;
        for (int c = 0; c < rank; ++c) ref[(size_t)s * rank + c] = 0.0;
        for (long long j = 0; j < m; ++j) {
            const float dx = P[i].x - P[j].x, dy = P[i].y - P[j].y, dz = P[i].z - P[j].z;
            const double g = exp2(-(double)fmaf(dz, dz, fmaf(dy, dy, dx * dx)));
            for (int c = 0; c < rank; ++c) ref[(size_t)s * rank + c] += g * X[(size_t)c * mpad + j];
        }
        for (int c = 0; c < rank; ++c) colscale[c] = fmax(colscale[c], fabs(ref[(size_t)s * rank + c]));
    }
    for (int s = 0; s < nsample; ++s)
        for (int c = 0; c < rank; ++c) {
            const double r = ref[(size_t)s * rank + c];
            en = fmax(en, fabs(on[(size_t)c * mpad + rowsel[s]] - r) / colscale[c]);
            if (time_old) eo = fmax(eo, fabs(oo[(size_t)c * mpad + rowsel[s]] - r) / colscale[c]);
        }
    printf("   accuracy on %d rows, per column relative to the column's largest sampled |value|: int8 digits %.3e   CUDA-core FP32 %.3e (%.3f ms)\n",
           nsample, en, eo, t_old);
    cudaFree(dY); cudaFree(dX); cudaFree(dOutNew); cudaFree(dOutOld); cudaFree(dPts); cudaFree(dPlanes); cudaFree(dPart); cudaFree(dColmax);
    return (en < 2e-6 || (time_old && en < 4.0 * eo + 1e-6) || xkind == 1) ? 0 : 4;      // xkind 1: fixed point vs a 5-decade column, reported only
}

int main(int argc, char** argv) {
    const long long m = argc > 1 ? atoll(argv[1]) : 50000;
    const int rank = argc > 2 ? atoi(argv[2]) : 200;
    const int rc = layout_tests_i8();
    printf("layout tests (i8, A in TMEM): %s\n", rc == 0 ? "PASS" : "FAIL");
    if (rc != 0) return rc;                     // 2: a wait timed out, the context is suspect; 3: a wrong layout, the products are too
    int rc2 = full_test_i8(3000, 200, 2.0, true, 0);
    if (rc2 == 2) return rc2;
    rc2 |= full_test_i8(20000, 230, 0.5, true, 1);
    rc2 |= full_test_i8(m, rank, 2.0, true, 0);
    printf("full tests (i8, A in TMEM): %s\n", rc2 == 0 ? "PASS" : "FAIL");
    return rc2;
}
