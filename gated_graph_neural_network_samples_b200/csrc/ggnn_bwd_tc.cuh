// Deterministic tensor-core (bf16x3) GEMMs of the propagation backward, sm_100a (tcgen05 / TMEM).  Selected with
// ggnn_set_backward_precision(GGNN_PREC_BF16X3); the fp32 FFMA kernels of ggnn_bwd.cuh stay the default.
//
// One kernel template computes   C (+)= sum_s op(A_s) . op(B_s)   with fp32 operands and fp32 results.  Every operand value is split
// x = hi + lo (two bf16, tc::split8) while it is written to shared memory, and every product is issued as 3 MMAs  hi.hi + hi.lo + lo.hi
// accumulating in fp32 in TMEM -- the arithmetic of the forward (ggnn_fwd_tc.cuh).  Two operand shapes:
//   NT (data gradients, every gemm_nt):   C[m, n] (+)= sum_s sum_k A[m, s*a_stride + k] . B[n, s*b_stride + k]
//        A, B row-major with K contiguous.  One CTA per 128 x NC output tile; the CTA runs the whole reduction (segments, then K) in a
//        fixed order, and its epilogue writes C or adds to it.
//   TN (weight gradients, every gemm_tn): C_s[k, n] += sum_m A_s[m, k] . B[m, n]
//        A_s, B row-major with the MMA's M (k) and N (n) dimensions contiguous.  The reduction over the nodes m is cut into S chunks
//        (S depends on the shape and the SM count only); every CTA writes its partial tile plainly into a workspace, and
//        tn_reduce_kernel adds the S partials to the caller's buffer in chunk order (S = 1: the epilogue adds directly).
//   Bias gradients (sum_m B[m, n]) are column sums of their own (colsum_part_kernel + colsum_det_kernel), whose order depends on M and N
//   only: a bias gradient has the same bits whether or not its kernel's gradient is requested.
// Either way a worker thread holds 8 K-consecutive values of one operand row, which it stores as one 16-byte core-matrix row of the
// canonical K-major no-swizzle layout the forward uses: no MN-major descriptors.  No float atomics anywhere: every result element is
// produced by one thread in a fixed order, so two calls on the same inputs give the same bits.
//
// Pipeline: 256 threads load the next K slab into registers while the tensor core works on the previous one; a ring of NSTAGE shared-
// memory stages, each owned by the whole CTA.  Thread 0 issues the MMAs of a stage and commits them to the stage's mbarrier; before a
// stage is rewritten, warp 0 alone waits (bounded) for the commit of its previous use and releases the others with __syncthreads.  A
// stage is rewritten only after its previous commit was observed, so no agent gets two phases ahead on a stage's barrier.
#pragma once
#include "ggnn_bwd.cuh"
#include "ggnn_fwd_tc.cuh"

namespace ggnn {
namespace bwdtc {

constexpr int BM = 128;          // UMMA M: output rows per CTA (NT: nodes, TN: rows of the weight gradient)
constexpr int BK = 32;           // reduction elements per stage (two UMMA K-steps)
constexpr int NSTAGE = 3;
constexpr int NTHREADS = 256;
constexpr int A_PART = BM * BK * 2;            // bytes of one bf16 part of an A stage (8 KB)
constexpr int A_STAGE = 2 * A_PART;            // hi + lo
constexpr int KGS_A = BM * 16;                 // byte stride between the 8-wide k-groups of an A stage
constexpr int MAX_NC = 256;

enum { MODE_NT = 0, MODE_TN = 1 };

struct TcGemmParams {
    // NT operands (K contiguous); TN's B operand ([M, N] row-major, N contiguous)
    const float* A; int lda; long long a_stride;
    const float* B; int ldb; long long b_stride;
    int nseg;
    bwd::SegList segs;         // TN: A_s, row-major [M, >= K] with row stride segs.ld[s]
    float* C; int ldc; long long c_stride;
    float* ws;                 // TN with S > 1: partial tiles [S][nseg][K][N]; nullptr: add into C
    int M, N, K;
    int nc;                    // N tile: power of two in [16, 256]
    int acc;                   // NT: add into C instead of overwriting it
    int rows_per_chunk;        // TN: nodes per reduction chunk (multiple of BK)
    int ktiles;                // TN: 128-row tiles of K
    int* error_flag;
};

__device__ __forceinline__ void ld8_k(const float* p, int kleft, float (&v)[8]) {   // 8 K-consecutive values, zero past the end (K % 4 == 0)
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (kleft >= 4) a = __ldg(reinterpret_cast<const float4*>(p));
    if (kleft >= 8) b = __ldg(reinterpret_cast<const float4*>(p + 4));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

template <int MODE>
__global__ void __launch_bounds__(NTHREADS) tc_gemm_kernel(const __grid_constant__ TcGemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar_mma[NSTAGE];
    __shared__ uint32_t s_tmem;
    __shared__ int s_abort;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NC = p.nc;
    const int B_PART = NC * BK * 2;
    const int STAGE = A_STAGE + 2 * B_PART;
    const int n0 = blockIdx.x * NC;
    // NT: rows m0.. of C, reduction over (segment, K).  TN: rows k0.. of C_seg, reduction over the nodes [mb, me) of one chunk.
    int m0 = 0, seg = 0, k0 = 0, mb = 0, me = 0, nit = 0, kslabs = 1;
    if (MODE == MODE_NT) {
        m0 = blockIdx.y * BM;
        kslabs = (p.K + BK - 1) / BK;
        nit = p.nseg * kslabs;
    } else {
        seg = blockIdx.y / p.ktiles;
        k0 = (blockIdx.y - seg * p.ktiles) * BM;
        mb = blockIdx.z * p.rows_per_chunk;
        me = min(p.M, mb + p.rows_per_chunk);
        nit = (me - mb + BK - 1) / BK;
    }
    const float* __restrict__ As = MODE == MODE_TN ? p.segs.p[seg] : p.A;
    const int lda = MODE == MODE_TN ? p.segs.ld[seg] : p.lda;

    if (tid == 0) {
        s_abort = 0;
        for (int i = 0; i < NSTAGE; ++i) tc::mbar_init(&bar_mma[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t tcols = NC < 32 ? 32u : (uint32_t)NC;   // power of two >= 32
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(&s_tmem)), "r"(tcols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = s_tmem;
    volatile int* abortp = &s_abort;

    // ---- register-staged loads: A stage = 128 rows x 4 k-groups (2 items per thread), B stage = NC rows x 4 k-groups (<= 4 per thread).
    // Item f: row = f % rows, k-group = f / rows -- consecutive lanes take consecutive rows, so the 16-byte shared stores never conflict.
    float ra[2][8], rb[4][8];
    auto load = [&](int it) {
        if (MODE == MODE_NT) {
            const int s = it / kslabs, kb = (it - s * kslabs) * BK;
            const float* Ag = p.A + (long long)s * p.a_stride;
            const float* Bg = p.B + (long long)s * p.b_stride;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int f = tid + j * NTHREADS, row = f & (BM - 1), kg = f >> 7;
                const int m = m0 + row, k = kb + kg * 8;
                ld8_k(Ag + (long long)m * p.lda + k, m < p.M ? p.K - k : 0, ra[j]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int f = tid + j * NTHREADS;
                const int row = f & (NC - 1), kg = f / NC;
                const int n = n0 + row, k = kb + kg * 8;
                ld8_k(Bg + (long long)n * p.ldb + k, (f < NC * 4 && n < p.N) ? p.K - k : 0, rb[j]);
            }
        } else {
            const int mbase = mb + it * BK;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int f = tid + j * NTHREADS, row = f & (BM - 1), kg = f >> 7;
                const int k = k0 + row, m = mbase + kg * 8;
                const bool ok = k < p.K;
#pragma unroll
                for (int i = 0; i < 8; ++i) ra[j][i] = (ok && m + i < me) ? __ldg(As + (long long)(m + i) * lda + k) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int f = tid + j * NTHREADS;
                const int row = f & (NC - 1), kg = f / NC;
                const int n = n0 + row, m = mbase + kg * 8;
                const bool ok = f < NC * 4 && n < p.N;
#pragma unroll
                for (int i = 0; i < 8; ++i) rb[j][i] = (ok && m + i < me) ? __ldg(p.B + (long long)(m + i) * p.ldb + n) : 0.f;
            }
        }
    };
    auto store = [&](int st) {
        uint8_t* a = smem + (size_t)st * STAGE;
        uint8_t* b = a + A_STAGE;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int f = tid + j * NTHREADS, row = f & (BM - 1), kg = f >> 7;
            uint4 hi, lo;
            tc::split8(ra[j], hi, lo);
            uint8_t* q = a + kg * KGS_A + row * 16;
            *reinterpret_cast<uint4*>(q) = hi;
            *reinterpret_cast<uint4*>(q + A_PART) = lo;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int f = tid + j * NTHREADS;
            if (f >= NC * 4) break;
            const int row = f & (NC - 1), kg = f / NC;
            uint4 hi, lo;
            tc::split8(rb[j], hi, lo);
            uint8_t* q = b + kg * (NC * 16) + row * 16;
            *reinterpret_cast<uint4*>(q) = hi;
            *reinterpret_cast<uint4*>(q + B_PART) = lo;
        }
    };
    // warp 0 waits for the commit that completes phase `phase` of stage `st`, everyone else waits behind the barrier
    auto wait_stage = [&](int st, int phase) -> bool {
        if (warp == 0 && !*abortp) {
            if (!tc::mbar_wait(&bar_mma[st], (uint32_t)(phase & 1), abortp)) *abortp = 1;
        }
        __syncthreads();
        return *abortp == 0;
    };

    const uint32_t idesc = tc::make_idesc_bf16(NC);
    if (nit > 0) load(0);
    bool ok = true;
    for (int it = 0; it < nit; ++it) {
        const int st = it % NSTAGE;
        if (it >= NSTAGE && !wait_stage(st, it / NSTAGE - 1)) { ok = false; break; }
        store(st);
        tc::fence_async_smem();
        tc::tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc::tc_fence_after();
            const uint32_t a_addr = tc::smem_u32(smem + (size_t)st * STAGE);
            const uint32_t b_addr = a_addr + A_STAGE;
#pragma unroll
            for (int ks = 0; ks < BK / 16; ++ks) {
                const uint64_t ah = tc::make_desc(a_addr + ks * 2 * KGS_A, KGS_A, 128), al = tc::make_desc(a_addr + ks * 2 * KGS_A + A_PART, KGS_A, 128);
                const uint64_t bh = tc::make_desc(b_addr + ks * 2 * NC * 16, NC * 16, 128), bl = tc::make_desc(b_addr + ks * 2 * NC * 16 + B_PART, NC * 16, 128);
                tc::umma_bf16(tmem, ah, bh, idesc, (it > 0 || ks > 0) ? 1u : 0u);
                tc::umma_bf16(tmem, ah, bl, idesc, 1u);
                tc::umma_bf16(tmem, al, bh, idesc, 1u);
            }
            tc::umma_commit(&bar_mma[st]);
        }
        if (it + 1 < nit) load(it + 1);   // global loads in flight while the MMAs run
    }
    // every stage's last commit has arrived (the final one implies all MMAs are complete) before TMEM is read and the CTA exits
    if (ok) {
        for (int st = 0; st < NSTAGE && st < nit; ++st) {
            const int last = st + (nit - 1 - st) / NSTAGE * NSTAGE;
            if (!wait_stage(st, last / NSTAGE)) { ok = false; break; }
        }
    }
    tc::tc_fence_after();

    if (ok) {
        // ---- epilogue: warp w reads TMEM lane quarter w % 4 (one output row per thread), column chunks of 8 alternate between w / 4 = 0, 1
        const int q = warp & 3, half = warp >> 2, row = q * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        float* dst = nullptr;
        bool add = false;
        if (MODE == MODE_NT) {
            const int m = m0 + row;
            if (m < p.M) dst = p.C + (long long)m * p.ldc;
            add = p.acc != 0;
        } else {
            const int k = k0 + row;
            if (k < p.K) {
                if (p.ws) dst = p.ws + (((long long)blockIdx.z * p.nseg + seg) * p.K + k) * p.N;
                else { dst = p.C + (long long)seg * p.c_stride + (long long)k * p.ldc; add = true; }
            }
        }
        for (int c = half; c < NC / 8; c += 2) {
            float v[8];
            if (nit > 0) tc::tmem_ld8(tmem + lane_addr + (uint32_t)(c * 8), v);
            else {
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = 0.f;
            }
            const int n = n0 + c * 8;
            if (dst) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (n + 4 * h + 4 > p.N) break;
                    float4* o = reinterpret_cast<float4*>(dst + n + 4 * h);
                    float4 x = make_float4(v[4 * h], v[4 * h + 1], v[4 * h + 2], v[4 * h + 3]);
                    if (add) { const float4 y = *o; x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w; }
                    *o = x;
                }
            }
        }
    }
    if (!ok && tid == 0) atomicExch(p.error_flag, 4);
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tcols) : "memory");
}

// C_s[k*ldc + n] += sum_{chunk} ws[chunk][s][k][n], chunks added in order
__global__ void __launch_bounds__(256) tn_reduce_kernel(const float* __restrict__ ws, int S, int nseg, int K, int N, float* __restrict__ C, int ldc,
                                                        long long c_stride) {
    const long long per = (long long)nseg * K * N;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < per; i += (long long)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int c = 0; c < S; ++c) s += ws[(long long)c * per + i];
        const long long sk = i / N;
        const int n = (int)(i - sk * N), sg = (int)(sk / K), k = (int)(sk - (long long)sg * K);
        C[sg * c_stride + (long long)k * ldc + n] += s;
    }
}

// part[chunk][n] = sum of src[m*ld + n] over the COLSUM_ROWS rows m of the chunk, in row order (one thread per column: coalesced)
constexpr int COLSUM_ROWS = 256;
__global__ void __launch_bounds__(256) colsum_part_kernel(const float* __restrict__ src, int ld, int M, int N, float* __restrict__ part) {
    const int n = blockIdx.x * 256 + threadIdx.x;
    if (n >= N) return;
    const int mb = blockIdx.y * COLSUM_ROWS, me = min(M, mb + COLSUM_ROWS);
    float s = 0.f;
    for (int m = mb; m < me; ++m) s += src[(long long)m * ld + n];
    part[(long long)blockIdx.y * N + n] = s;
}

// dst[n] += sum_{m < M} src[m*ld + n], one block per column, fixed per-thread strides and a fixed-shape tree: deterministic.
// (Second stage of the bias gradients, and the sum of the per-block partials of the attention weights' gradient.)
__global__ void __launch_bounds__(256) colsum_det_kernel(const float* __restrict__ src, int ld, int M, float* __restrict__ dst) {
    __shared__ float s[256];
    const int n = blockIdx.x;
    float a = 0.f;
    for (int m = threadIdx.x; m < M; m += 256) a += src[(long long)m * ld + n];
    s[threadIdx.x] = a;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) s[threadIdx.x] += s[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) dst[n] += s[0];
}

// ------------------------------------------------------------------------------------------------ host side
inline int pick_nc(int N) {
    if (N <= MAX_NC) { int nc = 16; while (nc < N) nc <<= 1; return nc; }
    const int pad256 = (N + 255) / 256 * 256 - N;
    return pad256 >= 128 ? 128 : 256;
}
inline size_t smem_bytes(int nc) { return (size_t)NSTAGE * (A_STAGE + 2 * (size_t)nc * BK * 2) + 1024; }

// Reduction chunks of a weight-gradient GEMM: enough CTAs to cover the SMs once, at least 256 nodes per chunk.
struct TnSplit { int S, rows_per_chunk, nc, ktiles; };
inline TnSplit tn_split(int M, int N, int K, int nseg, int num_sms) {
    TnSplit s;
    s.nc = pick_nc(N);
    s.ktiles = (K + BM - 1) / BM;
    const int tiles = ((N + s.nc - 1) / s.nc) * nseg * s.ktiles;
    int S = std::max(1, (num_sms + tiles - 1) / tiles);
    S = std::max(1, std::min(S, M / 256));
    int rpc = (M + S - 1) / S;
    rpc = (rpc + BK - 1) / BK * BK;
    s.rows_per_chunk = std::max(rpc, BK);
    s.S = (M + s.rows_per_chunk - 1) / s.rows_per_chunk;
    return s;
}
// workspace floats of that GEMM (0 when it adds into C directly)
inline size_t tn_workspace_floats(int M, int N, int K, int nseg, int num_sms) {
    const TnSplit s = tn_split(M, N, K, nseg, num_sms);
    return s.S > 1 ? (size_t)s.S * nseg * K * N : 0;
}

// raise the dynamic shared-memory limit of both instantiations on the current device (once per backward call)
inline cudaError_t configure_tc_gemm() {
    cudaError_t e = cudaFuncSetAttribute(tc_gemm_kernel<MODE_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(MAX_NC));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tc_gemm_kernel<MODE_TN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(MAX_NC));
    return e;
}

}  // namespace bwdtc
}  // namespace ggnn
