// tc_i8.cu - 5th-generation tensor cores (tcgen05, INT8 operands, INT32 accumulators in TMEM) for the rank update of
// the ICP posterior, M = I + A^T A (interpolatedModel.posterior, NonRigidIcpProposal.scala:152).
//
// The path is FP64 in the reference and tcgen05 has no FP64 kind, so the FP64 product is EMULATED exactly enough for the
// 1e-5 contract by split-integer arithmetic (Ozaki scheme): every column of A is scaled by a model-level bound into
// (-1/2, 1/2) and written as four balanced base-255 digits d_0..d_3 in [-127, 127] (int8 operands),
//     A[r][j] / s_j = sum_k d_k[r][j] 255^-(k+1) + O(255^-4),
// the digit matrices are multiplied on the tensor cores with exact INT32 accumulation (606 rows x 127^2 x 4 products
// < 2^31), digit pairs of equal weight k + l share one accumulator, and the four accumulators are recombined in FP64:
//     (A^T A)[i][j] = s_i s_j sum_t 255^-(t+2) ACC_t[i][j],   ACC_t = sum_{k+l=t} D_k^T D_l,  t = 0..3.
// Measured on the reference's femur GPMM-100 (tools/ozaki_study.py): max relative error of M 2e-9, of the posterior mean
// 1.4e-8 - three orders inside the 1e-5 contract, but not the 1e-9 the FP64 tensor-pipe path (DMMA) delivers, so this
// path is selected explicitly (ICPCUDA_RANK_UPDATE=int8).
//
// Both MMA operands are the SAME shared-memory image of a digit matrix (rows = the MMA's K dimension, columns = M resp. N),
// i.e. MN-major operands, which tcgen05 accepts for 8-bit types: no transposition anywhere.
//   canonical MN-major layout, no swizzle: 16 consecutive columns of one row = one 16-byte line; 8 consecutive rows = one
//   128-byte core matrix; core matrices tile the columns with stride SBO and the 8-row groups with stride LBO.
#include <algorithm>
#include <vector>

#include "icp_device.cuh"
#include "icp_internal.h"
#include "tc_ptx.cuh"

namespace icp {

// ---- PTX wrappers (CUDA 12.9, sm_100a) ----------------------------------------------------------------------------

// shared-memory matrix descriptor, SWIZZLE_NONE, version 1 (Blackwell): start address, leading (K-direction) and stride
// (MN-direction) byte offsets, all in units of 16 bytes
__device__ __forceinline__ uint64_t umma_desc_noswizzle(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// instruction descriptor of kind::i8: S32 accumulator, signed 8-bit A and B, both MN-major, M x N tile
__host__ __device__ constexpr uint32_t umma_idesc_i8(int M, int N) {
    return (2u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// 16 consecutive accumulator columns of this thread's TMEM lane (warp w of a warpgroup reads lanes 32 (w % 4) ..)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, int (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, int (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4_nowait(uint32_t taddr, int (&v)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// byte offset of the 16-byte line (row r, column chunk ch) inside a digit image: blocks of 32 rows (one MMA K step) of
// 4 KB, inside a block [row group of 8][chunk][row in group][16 bytes]  ->  SBO = 128, LBO = 1024
constexpr int kI8Cols = 128;          // columns of a digit image (MMA M; the first 112 are the MMA N)
constexpr int kI8N = 112;
constexpr int kI8BlockBytes = 32 * kI8Cols;
__device__ __forceinline__ uint32_t i8_line_offset(int r, int ch) {
    return (uint32_t)((r >> 5) * kI8BlockBytes + ((r & 31) >> 3) * 1024 + ch * 128 + (r & 7) * 16);
}

// ---- micro-benchmark / self-test: D = A^T A of one int8 matrix (rows x 128), `iters` passes over the same image ---------
__global__ void __launch_bounds__(128) k_i8_gram_test(int rows, const int8_t *__restrict__ A, int *__restrict__ D, int iters) {
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&s_tmem, 128);
    if (tid == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    const int nblk = rows / 32;
    for (int e = tid; e < rows * (kI8Cols / 16); e += blockDim.x) {
        const int r = e / (kI8Cols / 16), ch = e % (kI8Cols / 16);
        *reinterpret_cast<uint4 *>(smem + i8_line_offset(r, ch)) = *reinterpret_cast<const uint4 *>(A + (size_t)r * kI8Cols + ch * 16);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    if (tid == 0) {
        const uint32_t idesc = umma_idesc_i8(128, kI8N);
        for (int it = 0; it < iters; it++)
            for (int b = 0; b < nblk; b++) {
                const uint64_t desc = umma_desc_noswizzle(smem_u32(smem) + b * kI8BlockBytes, 1024, 128);
                umma_i8(tmem, desc, desc, idesc, (it | b) ? 1u : 0u);
            }
        umma_commit(&bar);
    }
    mbar_wait(&bar, 0);
    tc_fence_after();
    if (blockIdx.x == 0 && D) {
        for (int c0 = 0; c0 < kI8N; c0 += 16) {
            int v[16];
            tmem_ld16(tmem + ((uint32_t)(32 * warp) << 16) + c0, v);
#pragma unroll
            for (int k = 0; k < 16; k++) D[(size_t)(32 * warp + lane) * kI8Cols + c0 + k] = v[k];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

}  // namespace icp

using namespace icp;

extern "C" int32_t icp_debug_i8_gram(icp_ctx ctx, int32_t rows, const int8_t *A, int32_t *D, int32_t iters, int32_t ctas,
                                     double *ms) {
    icp_ctx _ctx = ctx;
    try {
        ICP_REQUIRE(ctx && A && rows >= 32 && rows % 32 == 0 && rows <= 1600 && iters >= 1 && ctas >= 1, "bad arguments");
        CtxLock lock(ctx);
        cudaStream_t s = ctx->stream;
        DevBuf<int8_t> dA;
        DevBuf<int> dD;
        dA.upload(A, (size_t)rows * kI8Cols, s);
        dD.alloc((size_t)kI8Cols * kI8Cols);
        ICP_CUDA(cudaMemsetAsync(dD.p, 0, sizeof(int) * kI8Cols * kI8Cols, s));
        const size_t smem = (size_t)rows * kI8Cols + 1024;
        ICP_CUDA(cudaFuncSetAttribute(k_i8_gram_test, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaEvent_t e0, e1;
        ICP_CUDA(cudaEventCreate(&e0));
        ICP_CUDA(cudaEventCreate(&e1));
        k_i8_gram_test<<<ctas, 128, smem, s>>>(rows, dA.p, dD.p, 1);       // warm-up + the checked result
        ICP_CUDA(cudaGetLastError());
        if (D) ICP_CUDA(cudaMemcpyAsync(D, dD.p, sizeof(int) * kI8Cols * kI8Cols, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        ICP_CUDA(cudaEventRecord(e0, s));
        k_i8_gram_test<<<ctas, 128, smem, s>>>(rows, dA.p, nullptr, iters);
        ICP_CUDA(cudaGetLastError());
        ICP_CUDA(cudaEventRecord(e1, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        float t = 0;
        ICP_CUDA(cudaEventElapsedTime(&t, e0, e1));
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        if (ms) *ms = t;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

// =======================================================================================================================
// Rank update of the ICP posterior on the INT8 tensor cores:  Mp = block-packed lower triangle of I + A^T A (+ Gs term),
// b = A^T y~.   Persistent, warp-specialised CTAs (one per SM: the four INT32 accumulators take all 512 TMEM columns),
// each walking its share of the chain-posteriors:
//
//   warp 14  "gather": per raw stage of 16 observations one TMA bulk copy (cp.async.bulk, mbarrier complete_tx) of the
//            observation's three unit-scaled basis rows (3 Kp doubles, contiguous in Qhat) into a ring in shared memory, and
//            the observation's whitening frame + right-hand side with cp.async (completion signalled on the same mbarrier)
//   warps 0..13  "converters": thread = (observation, 8 columns): the 3 x 3 whitening in FP64 straight into fixed point,
//            x = rn(f . Qhat * 2^30 / bound) (|x| <= 2^30), the four balanced base-256 digits of x are the bytes of
//            (x + 0x00808080) ^ 0x00808080, byte-transposed with PRMT into the four digit images of a 32-row MMA K block;
//            b accumulates in FP64 on the way
//   warp 15  "mma": one thread issues, per K block, the ten digit-pair products D_k^T D_l, k + l <= 3, into the accumulator
//            of weight 256^-(k+l) (tcgen05.mma kind::i8, both operands the same MN-major images), tcgen05.commit frees the
//            digit buffer for the converters
//   epilogue (all but the gather warp, which is already prefetching the next chain): tcgen05.ld, Horner in FP64 (exact:
//            |sum| < 2^53), scale by the column bounds, add I (+ the constant Gram term), write the 8 x 8 blocks
//            k_cholesky_packed consumes.
// Rows of A may be summed in any order (integer accumulation is exact), so K block d of a step holds frame row d of the
// step's 32 observations.
// =======================================================================================================================
namespace icp {

constexpr int kRuThreads = 512;
constexpr int kRuGatherWarp = 12, kRuMmaWarp = 15;    // the gather warp skips the epilogue: it sits in TMEM lane quarter 0, which has the fewest blocks
constexpr int kRuFrameDoubles = 14;                  // F (9), y (3), valid flag, pad: 112-byte stride = conflict-free LDS.128
constexpr int kRuRawObs = 16;                        // observations per raw stage

__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t *bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cp_async8(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16_cg(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
// executed by the whole (converged) warp with warp-uniform operands: one elected lane issues the copy
__device__ __forceinline__ void tma_bulk_g2s_elect(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "@p cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t"
        "}\n" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

#ifdef ICP_I8_TIMING
__device__ long long g_i8_timing[256 * 16];
#define I8T_DECL long long _tm[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long _t0 = clock64(), _tk = _t0; (void)_tk; (void)_tm;
#define I8T_MARK() (_tk = clock64())
#define I8T_ADD(i) do { const long long _n = clock64(); _tm[i] += _n - _tk; _tk = _n; } while (0)
#define I8T_FLUSH(cond, lo, hi) do { if (cond) for (int _i = lo; _i <= hi; _i++) g_i8_timing[(blockIdx.x & 255) * 16 + _i] = _tm[_i]; } while (0)
#else
#define I8T_DECL
#define I8T_MARK()
#define I8T_ADD(i)
#define I8T_FLUSH(cond, lo, hi)
#endif

struct I8Args {
    const double *Qhat;      // 3N x Kp: Q with every column divided by its bound colnorm_j (max over the vertices of |Q_v[:, j]|)
    const double *Qsub;      // nullable: the proposal's observation rows in slot order, [n][3 Kp + 2] (= the shared-memory stride):
                             // one bulk copy per raw stage instead of one per observation (every slot is then an observation)
    const double *colnorm;   // Kp (0 on the padding)
    double fmul;             // frame rows are multiplied by this: |fmul * F_d . Qhat_v[:, j]| <= 2^30
    double w2;               // (A^T A)[i][j] = colnorm_i colnorm_j w2 * sum_t 256^(3-t) ACC_t[i][j]
    double bscale;           // b_j = colnorm_j bscale * (accumulated value)
    int nraw;                // raw stages in the ring
};

// digit buffer geometry: K block = 4 row groups of 8 rows; a row group holds the 4 images' 7 column chunks side by side
// (28 chunks + 1 pad chunk of 128 B), so that an MMA's B operand can span two adjacent images (N = 224)
constexpr int kRuChunksPerImage = 7;                 // 112 columns
constexpr int kRuGroupBytes = (4 * kRuChunksPerImage + 1) * 128;   // 3712
constexpr int kRuKBlockBytes = 4 * kRuGroupBytes;                  // 14848
constexpr int kRuAccStride = 112;                    // TMEM columns between the accumulators of consecutive weights

// observation row of rank-update entry e (ObsDev::list, ObsDev::row)
__device__ __forceinline__ int obs_row(const ObsDev &o, int e) {
    const int c = o.list ? __ldg(o.list + e) : e;
    return o.row ? __ldg(o.row + c) : c;
}

template <int RPO>
__global__ void __launch_bounds__(kRuThreads, 1) k_rank_update_i8(ModelDev m, ObsDev o, int C, I8Args a, const double *__restrict__ Gs,
                                                                  double gs_scale, double *__restrict__ Mp,
                                                                  double *__restrict__ bvec) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int kBufBytes = RPO * kRuKBlockBytes;             // one digit buffer: RPO K blocks of 32 rows
    __shared__ uint64_t full_raw[8], empty_raw[8], full_dig[2], empty_dig[2], acc_done;
    __shared__ uint32_t s_tmem;
    __shared__ int s_poison[3];        // by chain % 3: written a chain early by the converters' look-ahead step
    const int Kp = m.Kp, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NG = Kp >> 3, NPAIR = (NG + 1) >> 1, ncv = 2 * NPAIR;      // column groups of 8, converter warps
    const int row_bytes = Kp * 8, obs_bytes = 3 * row_bytes, obs_stride = obs_bytes + 16;
    const int raw_stage = kRuRawObs * obs_stride, NRAW = a.nraw;
    unsigned char *dig = smem;
    unsigned char *raw = smem + ((2 * kBufBytes + 127) & ~127);
    double *frames = reinterpret_cast<double *>(raw + (size_t)NRAW * raw_stage);     // [NRAW][16][14]
    double *s_b = frames + (size_t)NRAW * kRuRawObs * kRuFrameDoubles;                // [2 chains in flight][2 teams][Kp]
    double *s_cn = s_b + 4 * Kp;                                                     // [128]
    double *s_gs = s_cn + 128;                                                       // RPO == 1: gs_scale * Gs, block-packed like Mp
    if (warp == 0) tmem_alloc(&s_tmem, 512);
    if (tid == 0) {
        for (int i = 0; i < NRAW; i++) { mbar_init(&full_raw[i], 32 + kRuRawObs); mbar_init(&empty_raw[i], NPAIR); }
        for (int i = 0; i < 2; i++) { mbar_init(&full_dig[i], NPAIR); mbar_init(&empty_dig[i], 1); }
        mbar_init(&acc_done, 1);
        s_poison[0] = s_poison[1] = s_poison[2] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int j = tid; j < 128; j += kRuThreads) s_cn[j] = j < Kp ? a.colnorm[j] : 0.0;
    if (RPO == 1) {
        const int NB = Kp >> 3;
        for (int e = tid; e < NB * (NB + 1) / 2 * 64; e += kRuThreads) {
            const int blk = e >> 6, r = (e >> 3) & 7, cc = e & 7;
            int bi = (int)((sqrtf(8.f * blk + 1.f) - 1.f) * 0.5f);
            while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
            while (bi * (bi + 1) / 2 > blk) bi--;
            const int bj = blk - bi * (bi + 1) / 2;
            s_gs[e] = gs_scale * Gs[(size_t)(8 * bi + r) * Kp + 8 * bj + cc];
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const int nmax = o.n;
    if (o.count) C = min(C, *o.count);   // list form: the entries of this launch (M / b of entry e are written at e)
    I8T_DECL

    if (warp == kRuGatherWarp) {
        // ---------------- gather warp: raw stage R of the CTA's flattened (chain, stage) sequence ----------------
        unsigned R = 0, slot = 0, gphase = 0;                  // stage counter, its ring slot and the parity of R / NRAW
        int c = blockIdx.x, rc = c < C ? obs_row(o, c) : 0;    // entry c, its observation row rc
        int nrows = c < C ? (o.nrows ? min(o.nrows[rc], nmax) : nmax) : 0;
        int nst = 2 * ((nrows + 31) >> 5), rs = 0;
        while (c < C && nst == 0) {
            c += gridDim.x;
            rc = c < C ? obs_row(o, c) : 0;
            nrows = c < C ? (o.nrows ? min(o.nrows[rc], nmax) : nmax) : 0;
            nst = 2 * ((nrows + 31) >> 5);
        }
        int v = -1;                                             // vertex of (c, rs) of lane's observation, loaded one stage ahead
        if (c < C && lane < kRuRawObs && lane < nrows) v = __ldg(o.vid + (size_t)rc * nmax + lane);
        while (c < C) {
            // successor (c2, rs2)
            int c2 = c, rc2 = rc, rs2 = rs + 1, nrows2 = nrows, nst2 = nst;
            if (rs2 >= nst) {
                rs2 = 0;
                do {
                    c2 += gridDim.x;
                    rc2 = c2 < C ? obs_row(o, c2) : 0;
                    nrows2 = c2 < C ? (o.nrows ? min(o.nrows[rc2], nmax) : nmax) : 0;
                    nst2 = 2 * ((nrows2 + 31) >> 5);
                } while (c2 < C && nst2 == 0);
            }
            int vnext = -1;
            if (c2 < C && lane < kRuRawObs && rs2 * kRuRawObs + lane < nrows2) vnext = __ldg(o.vid + (size_t)rc2 * nmax + rs2 * kRuRawObs + lane);
            I8T_MARK();
            if (R >= (unsigned)NRAW) mbar_wait(&empty_raw[slot], gphase ^ 1u);      // parity of use (R / NRAW) - 1
            I8T_ADD(7);
            const int g0 = rs * kRuRawObs, nob = max(0, min(kRuRawObs, nrows - g0));       // observation slots of this stage
            double *fr0 = frames + (size_t)slot * kRuRawObs * kRuFrameDoubles;
            {   // frames and right-hand sides: 9 nob + 3 nob contiguous doubles, dealt over the 32 lanes
                const double *F = o.F + ((size_t)rc * nmax + g0) * 9, *y = o.y + ((size_t)rc * nmax + g0) * 3;
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    const int e = lane + 32 * j;
                    if (e < 9 * nob) cp_async8(fr0 + (e / 9) * kRuFrameDoubles + e % 9, F + e);
                }
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const int e = lane + 32 * j;
                    if (e < 3 * nob) cp_async8(fr0 + (e / 3) * kRuFrameDoubles + 9 + e % 3, y + e);
                }
                cp_async_mbar_arrive_noinc(&full_raw[slot]);
            }
            if (lane < kRuRawObs) fr0[lane * kRuFrameDoubles + 12] = v >= 0 ? 1.0 : 0.0;
            const uint32_t dst = smem_u32(raw + (size_t)slot * raw_stage), bar = smem_u32(&full_raw[slot]);
            const bool leader = lane == 0;
            if (a.Qsub) {
                // every slot of the stage is an observation: one bulk copy
                if (leader && nob > 0) {
                    mbar_arrive_expect_tx(&full_raw[slot], (uint32_t)(nob * obs_stride));
                    tma_bulk_g2s_u32(dst, reinterpret_cast<const unsigned char *>(a.Qsub) + (size_t)g0 * obs_stride, (uint32_t)(nob * obs_stride), bar);
                } else if (lane < kRuRawObs) mbar_arrive(&full_raw[slot]);
            } else {
                // one bulk copy per observation (3 Kp doubles, contiguous in Qhat). Measured alternatives, all slower than the
                // compiler's per-lane issue loop (~77 clocks per copy): straight-line issue from warp-uniform operands
                // (redux + elect.sync, ~130 clocks per copy) and 16-byte cp.async.cg dealt over the lanes (~330 clocks per row triple)
                if (lane < kRuRawObs) {
                    if (v >= 0) {
                        mbar_arrive_expect_tx(&full_raw[slot], (uint32_t)obs_bytes);
                        tma_bulk_g2s_u32(dst + (uint32_t)(lane * obs_stride), a.Qhat + (size_t)3 * v * Kp, (uint32_t)obs_bytes, bar);
                    } else mbar_arrive(&full_raw[slot]);
                }
            }
            __syncwarp();
            I8T_ADD(8);
            R++;
            if (++slot == (unsigned)NRAW) { slot = 0; gphase ^= 1u; }                   // (no integer division in the loops: R % NRAW and
                                                                                        //  R / NRAW cost ~700 clocks per stage under contention)
            c = c2; rc = rc2; rs = rs2; nrows = nrows2; nst = nst2; v = vnext;
        }
        I8T_FLUSH(lane == 0, 7, 8);
    } else {
        unsigned S = 0, it = 0, nacc = 0;                        // 32-observation steps / chains / non-empty chains done by this CTA
        // converter state
        const int cw = warp < kRuGatherWarp ? warp : warp - 1;       // converter index 0..13 (warps 0..11, 13, 14)
        const int pair = cw >> 1, h = cw & 1, gh = (lane >> 3) & 1, g = 2 * pair + gh;
        const int osl = (lane & 7) + 8 * (lane >> 4);                 // observation inside the raw stage (0..15)
        const bool live = cw < ncv && g < NG;
        double bacc[8];
#pragma unroll
        for (int k = 0; k < 8; k++) bacc[k] = 0.0;
        bool ovf = false;
        int pre_done = 0;                                             // the team's first step of this chain was converted early
        // ring slot and use parity of the team's next raw stage R = 2 Sg + pass: the team converts every other 32-observation
        // step, in order, so R advances by 1, 3, 1, 3, ... - kept incrementally, no integer division in the loop
        unsigned rslot = (2u * (unsigned)h) % (unsigned)NRAW, rphase = ((2u * (unsigned)h) / (unsigned)NRAW) & 1u;
        auto advance = [&](unsigned k) { rslot += k; while (rslot >= (unsigned)NRAW) { rslot -= (unsigned)NRAW; rphase ^= 1u; } };
        auto reduce_b = [&]() {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                double s = bacc[k];
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                s += __shfl_xor_sync(0xffffffffu, s, 4);
                s += __shfl_xor_sync(0xffffffffu, s, 16);
                bacc[k] = s;
            }
        };
        // one 32-observation step (global index Sg) of team h: two raw stages of 16 observations into digit buffer h
        auto convert_step = [&](unsigned Sg) {
            const double lim = 1.152921504606846976e18;               // 2^60: |fmul F_d|^2 above it could leave |x| <= 2^30
#pragma unroll 1
            for (int pass = 0; pass < 2; pass++) {
                const unsigned slot = rslot;
                I8T_MARK();
                mbar_wait(&full_raw[slot], rphase);
                I8T_ADD(1);
                advance(pass == 0 ? 1u : 3u);
                const double *fr = frames + ((size_t)slot * kRuRawObs + osl) * kRuFrameDoubles;
                const bool valid = live && fr[12] != 0.0;
                double f[12];
                double2 q[3][4];
                if (valid) {
#pragma unroll
                    for (int k = 0; k < 6; k++) { const double2 t2 = reinterpret_cast<const double2 *>(fr)[k]; f[2 * k] = t2.x; f[2 * k + 1] = t2.y; }
                    const unsigned char *rp = raw + (size_t)slot * raw_stage + (size_t)osl * obs_stride + g * 64;
#pragma unroll
                    for (int d = 0; d < 3; d++)
#pragma unroll
                        for (int k = 0; k < 4; k++) q[d][k] = *reinterpret_cast<const double2 *>(rp + d * row_bytes + 16 * k);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_raw[slot]);             // NPAIR warps read this stage: one arrival each
                I8T_ADD(12);
                if (pass == 0 && Sg >= 2) mbar_wait(&empty_dig[h], ((Sg >> 1) - 1) & 1);
                I8T_ADD(2);
                // 16-byte line of (row 16 pass + osl, image 0, chunk pair) inside a K block, + this thread's 8-byte half
                unsigned char *blk = dig + h * kBufBytes + (2 * pass + (lane >> 4)) * kRuGroupBytes + pair * 128 + (lane & 7) * 16 + gh * 8;
                if (valid) {
                    double w0 = 0, w1 = 0, w2v = 0;
                    if (RPO == 1) {
                        // b += Q_i^T (F^T F y)
                        w0 = f[0] * f[9] + f[3] * f[10] + f[6] * f[11];
                        w1 = f[1] * f[9] + f[4] * f[10] + f[7] * f[11];
                        w2v = f[2] * f[9] + f[5] * f[10] + f[8] * f[11];
                    }
#pragma unroll
                    for (int d = 0; d < RPO; d++) {
                        const double f0 = f[3 * d] * a.fmul, f1 = f[3 * d + 1] * a.fmul, f2 = f[3 * d + 2] * a.fmul;
                        ovf = ovf || !(fma(f2, f2, fma(f1, f1, f0 * f0)) <= lim);        // also catches NaN frames
                        uint32_t w[8];
#pragma unroll
                        for (int k = 0; k < 8; k++) {
                            const double qa = (k & 1) ? q[0][k >> 1].y : q[0][k >> 1].x, qb = (k & 1) ? q[1][k >> 1].y : q[1][k >> 1].x,
                                         qc = (k & 1) ? q[2][k >> 1].y : q[2][k >> 1].x;
                            const double av = fma(f2, qc, fma(f1, qb, f0 * qa));
                            if (RPO == 3) bacc[k] = fma(f[9 + d], av, bacc[k]);
                            else bacc[k] = fma(w0, qa, fma(w1, qb, fma(w2v, qc, bacc[k])));
                            // x = rn(av) (|av| <= 2^30) is the low word of av + 1.5 * 2^52; the constant also carries the
                            // + 0x00808080 of the balanced base-256 digits: x + 0x00808080 = sum_k (d_k + 128 [k > 0]) 256^(3-k)
                            w[k] = (uint32_t)__double2loint(av + (6755399441055744.0 + 8421504.0));
                        }
                        // 4 x 4 byte transposes: image q gets byte 3 - q of the eight words; the lower digits leave their
                        // + 128 offset here (^ 0x80 per byte), the top byte is the signed leading digit as it is
                        const uint32_t t0 = prmt(w[0], w[1], 0x5140), t1 = prmt(w[0], w[1], 0x7362), t2 = prmt(w[2], w[3], 0x5140),
                                       t3 = prmt(w[2], w[3], 0x7362), u0 = prmt(w[4], w[5], 0x5140), u1 = prmt(w[4], w[5], 0x7362),
                                       u2 = prmt(w[6], w[7], 0x5140), u3 = prmt(w[6], w[7], 0x7362);
                        unsigned char *bd = blk + d * kRuKBlockBytes;
                        const uint32_t X = 0x80808080u;
                        *reinterpret_cast<uint2 *>(bd + 3 * kRuChunksPerImage * 128) = make_uint2(prmt(t0, t2, 0x5410) ^ X, prmt(u0, u2, 0x5410) ^ X);
                        *reinterpret_cast<uint2 *>(bd + 2 * kRuChunksPerImage * 128) = make_uint2(prmt(t0, t2, 0x7632) ^ X, prmt(u0, u2, 0x7632) ^ X);
                        *reinterpret_cast<uint2 *>(bd + 1 * kRuChunksPerImage * 128) = make_uint2(prmt(t1, t3, 0x5410) ^ X, prmt(u1, u3, 0x5410) ^ X);
                        *reinterpret_cast<uint2 *>(bd) = make_uint2(prmt(t1, t3, 0x7632), prmt(u1, u3, 0x7632));
                    }
                } else if (live) {
#pragma unroll
                    for (int d = 0; d < RPO; d++)
#pragma unroll
                        for (int qq = 0; qq < 4; qq++)
                            *reinterpret_cast<uint2 *>(blk + d * kRuKBlockBytes + qq * kRuChunksPerImage * 128) = make_uint2(0u, 0u);
                }
                I8T_ADD(3);
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_dig[h]);
            I8T_ADD(13);
        };
        for (int c = blockIdx.x; c < C; c += gridDim.x, it++) {
            const int nrows = o.nrows ? min(o.nrows[obs_row(o, c)], nmax) : nmax;
            const int nsteps = (nrows + 31) >> 5;
            double *sb = s_b + (it & 1) * 2 * Kp;
            if (warp == kRuMmaWarp) {
                // ---------------- MMA warp ----------------
                const uint32_t idw = umma_idesc_i8(128, 2 * kRuAccStride), idn = umma_idesc_i8(128, kRuAccStride);
                for (int st = 0; st < nsteps; st++) {
                    const unsigned Sg = S + st, buf = Sg & 1;
                    I8T_MARK();
                    mbar_wait(&full_dig[buf], (Sg >> 1) & 1);
                    I8T_ADD(5);
                    tc_fence_after();
                    if (lane == 0) {
                        const uint32_t sbase = smem_u32(dig + buf * kBufBytes);
#pragma unroll 1
                        for (int d = 0; d < RPO; d++) {
                            // image q of K block d: operand descriptors start at its first chunk; LBO = row-group stride
                            auto img = [&](int q) { return umma_desc_noswizzle(sbase + d * kRuKBlockBytes + q * kRuChunksPerImage * 128, kRuGroupBytes, 128); };
                            const uint32_t first = (st | d) ? 1u : 0u;
                            // D_k^T [D_l D_l+1] lands in the accumulators of weight k + l and k + l + 1 (adjacent TMEM columns)
                            umma_i8(tmem + 0 * kRuAccStride, img(0), img(0), idw, first);     // (0,0) (0,1)
                            umma_i8(tmem + 2 * kRuAccStride, img(0), img(2), idw, first);     // (0,2) (0,3)
                            umma_i8(tmem + 1 * kRuAccStride, img(1), img(0), idw, 1u);        // (1,0) (1,1)
                            umma_i8(tmem + 3 * kRuAccStride, img(1), img(2), idn, 1u);        // (1,2)
                            umma_i8(tmem + 2 * kRuAccStride, img(2), img(0), idw, 1u);        // (2,0) (2,1)
                            umma_i8(tmem + 3 * kRuAccStride, img(3), img(0), idn, 1u);        // (3,0)
                        }
                        umma_commit(&empty_dig[buf]);
                        if (st == nsteps - 1) umma_commit(&acc_done);
                    }
                    __syncwarp();
                    I8T_ADD(6);
                }
            } else if (cw < ncv) {
                // ---------------- converter warps: team h = cw & 1 converts the steps of its parity into digit buffer h ----------------
                // steps of this chain the team still owes, then - while the tensor core finishes the chain - its first step
                // of the next chain (one call site of the step body: two would double its register footprint)
                int st = ((h - (int)S) & 1) + 2 * pre_done;
                // the team's first step of every chain is reduced and parked in shared memory on its own, whether it ran early
                // (the previous chain's tail) or runs here: b then sums in the same order in every chain, so a chain's b does not
                // depend on whether it is the first chain of its CTA
                bool had_pre = pre_done != 0;
                pre_done = 0;
                bool published = false;
                for (;;) {
                    unsigned Sg;
                    if (st < nsteps) { Sg = S + st; st += 2; }
                    else if (!published) {
                        // b: the 16 observation lanes of this warp (same gh), fixed order; the two teams meet in shared memory.
                        // The early step's share is already there (it must not stay in registers across the epilogue)
                        reduce_b();
                        if (live && (lane & 23) == 0) {                       // lanes 0 and 8: one per column group
#pragma unroll
                            for (int k = 0; k < 8; k++) sb[h * Kp + 8 * g + k] = bacc[k] + (had_pre ? sb[h * Kp + 8 * g + k] : 0.0);
                        }
                        if (__any_sync(0xffffffffu, ovf) && lane == 0) atomicOr(&s_poison[it % 3], 1);
                        ovf = false;
#pragma unroll
                        for (int k = 0; k < 8; k++) bacc[k] = 0.0;
                        published = true;
                        const int c2 = c + gridDim.x;
                        if (c2 >= C) break;
                        const int nrows2 = o.nrows ? min(o.nrows[obs_row(o, c2)], nmax) : nmax, nsteps2 = (nrows2 + 31) >> 5;
                        const unsigned S2 = S + nsteps;
                        const int first2 = (h - (int)S2) & 1;
                        if (first2 >= nsteps2) break;
                        Sg = S2 + first2;
                        pre_done = 1;
                    } else break;
                    convert_step(Sg);
                    if (published) break;
                    if (!had_pre) {
                        reduce_b();
                        if (live && (lane & 23) == 0) {
#pragma unroll
                            for (int k = 0; k < 8; k++) sb[h * Kp + 8 * g + k] = bacc[k];
                        }
#pragma unroll
                        for (int k = 0; k < 8; k++) bacc[k] = 0.0;
                        had_pre = true;
                    }
                }
                if (pre_done) {
                    // the early step's share of the next chain's b goes to that chain's buffer now
                    reduce_b();
                    double *sbn = s_b + ((it + 1) & 1) * 2 * Kp;
                    if (live && (lane & 23) == 0) {
#pragma unroll
                        for (int k = 0; k < 8; k++) sbn[h * Kp + 8 * g + k] = bacc[k];
                    }
#pragma unroll
                    for (int k = 0; k < 8; k++) bacc[k] = 0.0;
                    if (__any_sync(0xffffffffu, ovf) && lane == 0) atomicOr(&s_poison[(it + 1) % 3], 1);
                    ovf = false;
                }
                I8T_MARK();
            }
            S += nsteps;
            // ---------------- epilogue: every warp but the gather warp ----------------
            named_bar_sync(1, kRuThreads - 32);
            I8T_ADD(4);
            const bool bad = s_poison[it % 3] != 0;
            for (int j = tid; j < Kp; j += kRuThreads)
                bvec[(size_t)c * Kp + j] = bad ? NAN : (sb[j] + sb[Kp + j]) * s_cn[j] * a.bscale;
            I8T_MARK();
            if (nsteps > 0) { mbar_wait(&acc_done, nacc & 1); nacc++; }
            I8T_ADD(9);
            tc_fence_after();
            {
                // warp = TMEM lane quarter qd (rows 32 qd ..); the half blocks (4 columns) of the 8-column blocks bj <= 4 qd + 3 are
                // dealt over the quarter's warps (16 accumulator registers per task: nothing of the converters' state spills)
                const int qd = warp & 3, i = 32 * qd + lane, NB = Kp >> 3, ntri = NB * (NB + 1) / 2;
                const int nw = qd == (kRuGatherWarp & 3) ? 3 : 4, idx = warp >> 2;          // (quarter 0's missing warp is its last: idx stays dense)
                const int nhalf = 2 * min(4 * qd + 4, NB);
                double *Mc = Mp + (size_t)c * ntri * 64;
                const double cij = (i < Kp && nsteps > 0) ? s_cn[i] * a.w2 : 0.0;   // no observation: the accumulators are undefined
                const int bi = i >> 3;
                if (32 * qd < Kp)
                    for (int hb = idx; hb < nhalf; hb += nw) {
                        // (two half blocks in flight - the next one's TMEM loads issued before this one's arithmetic - needs 16 more
                        // registers, spills, and measured 2.7x slower: with 220 KB of shared memory the L1 is too small for local memory)
                        const int bj = hb >> 1, j0 = 4 * hb;
                        int a0[4], a1[4], a2[4], a3[4];
                        const uint32_t ta = tmem + ((uint32_t)(32 * qd) << 16) + j0;
                        tmem_ld4_nowait(ta, a0); tmem_ld4_nowait(ta + kRuAccStride, a1); tmem_ld4_nowait(ta + 2 * kRuAccStride, a2);
                        tmem_ld4_nowait(ta + 3 * kRuAccStride, a3);
                        tmem_ld_wait();
                        if (i < Kp && bj <= bi) {
                            const int off = ((bi * (bi + 1) >> 1) + bj) * 64 + (i & 7) * 8 + (j0 & 7);
                            double *dst = Mc + off;
#pragma unroll
                            for (int k = 0; k < 4; k += 2) {
                                double vv[2];
#pragma unroll
                                for (int u = 0; u < 2; u++) {
                                    const int kk = k + u, j = j0 + kk;
                                    // exact integer Horner in base 256 (|H| < 2^51), then int64 -> double through the 1.5 * 2^52 offset
                                    const long long H = (((long long)a0[kk] * 256 + a1[kk]) * 256 + a2[kk]) * 256 + a3[kk];
                                    const double acc = __longlong_as_double(H + 0x4338000000000000ll) - 6755399441055744.0;
                                    double val = fma(cij * s_cn[j], acc, i == j ? 1.0 : 0.0);
                                    if (RPO == 1) val += s_gs[off + kk];
                                    vv[u] = bad ? NAN : val;
                                }
                                __stcs(reinterpret_cast<double2 *>(dst + k), make_double2(vv[0], vv[1]));
                            }
                        }
                    }
            }
            I8T_ADD(14);
            tc_fence_before();
            named_bar_sync(1, kRuThreads - 32);
            tc_fence_after();
            if (tid == 0) s_poison[it % 3] = 0;     // next written for chain it + 3, at the earliest after the barriers of chain it + 1
            I8T_ADD(10);
#ifdef ICP_I8_TIMING
            _tm[11] += 1;
#endif
        }
        I8T_FLUSH(tid == 0, 1, 4);
        I8T_FLUSH(tid == 0, 9, 14);
#ifdef ICP_I8_TIMING
        if (warp == 3) { _tm[15] = _tm[14]; I8T_FLUSH(lane == 0, 15, 15); }
#endif
        I8T_FLUSH(warp == kRuMmaWarp && lane == 0, 5, 6);
    }
#ifdef ICP_I8_TIMING
    if (tid == 0) g_i8_timing[(blockIdx.x & 255) * 16] = clock64() - _t0;
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// the observation rows of a model-sampling proposal in slot order, padded to the shared-memory stride of the rank update
__global__ void k_pack_obs_rows(int n, int Kp, const int *__restrict__ ids, const double *__restrict__ Qhat, double *__restrict__ Qsub) {
    const int i = blockIdx.x, stride = 3 * Kp + 2;
    const double *src = Qhat + (size_t)3 * ids[i] * Kp;
    for (int e = threadIdx.x; e < stride; e += blockDim.x) Qsub[(size_t)i * stride + e] = e < 3 * Kp ? src[e] : 0.0;
}
void launch_pack_obs_rows(int n, int Kp, const int *d_ids, const double *d_Qhat, double *d_Qsub, cudaStream_t s) {
    if (n <= 0) return;
    k_pack_obs_rows<<<n, 128, 0, s>>>(n, Kp, d_ids, d_Qhat, d_Qsub);
    ICP_CUDA(cudaGetLastError());
}

__global__ void k_unit_basis(long long total, int Kp, const double *__restrict__ Q, const double *__restrict__ colnorm, double *__restrict__ Qhat) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    const double cn = colnorm[g % Kp];
    Qhat[g] = cn > 0.0 ? Q[g] / cn : 0.0;
}
void launch_unit_basis(int rows, int Kp, const double *d_Q, const double *d_colnorm, double *d_Qhat, cudaStream_t s) {
    const long long total = (long long)rows * Kp;
    k_unit_basis<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(total, Kp, d_Q, d_colnorm, d_Qhat);
    ICP_CUDA(cudaGetLastError());
}

}  // namespace icp
#ifdef ICP_I8_TIMING
extern "C" int32_t icp_debug_i8_timing(long long *out, int32_t n) {
    return (int32_t)cudaMemcpyFromSymbol(out, icp::g_i8_timing, sizeof(long long) * std::min(n, 256 * 16));
}
#endif
namespace icp {
// false: outside the kernel's domain (nothing launched) - the caller takes the FP64 tensor-pipe path
bool launch_rank_update_i8(const ModelDev &m, int C, const ObsDev &o, const GramFast *gf, const I8Model &im, const I8Scale &sc,
                           double *d_Mp, double *d_b, int n_sm, cudaStream_t s) {
    const int rpo = gf ? 1 : 3;
    // INT32 accumulators: rows * 4 digit pairs * 128^2 < 2^31
    if (C <= 0 || m.Kp > kI8N || (m.Kp & 7) || !im.Qhat || (long long)o.n * rpo > 32000 || !(sc.fmul > 0.0) || !std::isfinite(sc.fmul)) return false;
    ProfScope _ps(ST_POSTERIOR_BUILD, s);
    const size_t obs_stride = (size_t)3 * m.Kp * 8 + 16;
    const size_t per_stage = kRuRawObs * obs_stride + kRuRawObs * kRuFrameDoubles * 8;
    const size_t fixed = (size_t)2 * rpo * kRuKBlockBytes + 128 + (size_t)(4 * m.Kp + 128) * 8 + 1024 +
                         (gf ? (size_t)(m.Kp / 8) * (m.Kp / 8 + 1) / 2 * 64 * 8 : 0);
    const size_t budget = 227 * 1024 - 1024;     // static shared memory (barriers) comes on top
    int nraw = (int)std::min<size_t>(8, (budget - fixed) / per_stage);
    if (nraw < 2) return false;
    I8Args a{im.Qhat, gf ? im.Qsub : nullptr, im.colnorm, sc.fmul, sc.w2, sc.bscale, nraw};
    // one CTA per SM (all 512 TMEM columns): ask for more than half of the shared memory so that no second CTA is scheduled
    // only to wait for the allocation
    const size_t smem = std::max<size_t>(fixed + nraw * per_stage, 120 * 1024);
    const int grid = std::min(C, std::max(1, n_sm));
    if (gf) {
        ICP_CUDA(cudaFuncSetAttribute(k_rank_update_i8<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_rank_update_i8<1><<<grid, kRuThreads, smem, s>>>(m, o, C, a, gf->Gs, gf->gs_scale, d_Mp, d_b);
    } else {
        ICP_CUDA(cudaFuncSetAttribute(k_rank_update_i8<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_rank_update_i8<3><<<grid, kRuThreads, smem, s>>>(m, o, C, a, nullptr, 0.0, d_Mp, d_b);
    }
    ICP_CUDA(cudaGetLastError());
    return true;
}

}  // namespace icp
