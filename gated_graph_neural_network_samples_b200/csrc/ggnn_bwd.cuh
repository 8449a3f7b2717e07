// Backward of the GGNN propagation step (what optimizer.compute_gradients builds for sparse:117-218 / dense:93-117,
// chem_tensorflow.py:184), fp32 on CUDA cores.  Per timestep, in reverse, with the activations the forward saved
// (state entering the step h, aggregated messages x, gates r/u, candidate c):
//
//   GRU :  dc = dh'*(1-u)   du = dh'*(h-c)   dh = dh'*u
//          dpc = dc*act'(c)        d[res..,x,rh] = dpc . K_c^T     dK_c += [res..,x,rh]^T . dpc     db_c += sum dpc
//          dr = drh*h   dh += drh*r   dpr = dr*r(1-r)   dpu = du*u(1-u)
//          d[res..,x,h] += [dpr|dpu] . K_g^T                       dK_g += [res..,x,h]^T . [dpr|dpu]  db_g += sum
//   RNN :  dpc = dh'*act'(h')      d[res..,x,h] = dpc . K^T        dK += [res..,x,h]^T . dpc          db += sum dpc
//   CudnnCompatibleGRUCell: dpc as GRU;  d[res..,x] = dpc . K_in^T   dK_in += [res..,x]^T . dpc   db_in += sum dpc
//          dq = dpc*r   dh += dq . K_hid^T   dK_hid += h^T . dq   db_hid += sum dq   dpr = dpc*q*r(1-r)   gates as GRU
//   msgs:  dx' = dx / (deg+1e-7)   dB[t] += sum_v indeg[v,t] dx'[v]
//          dW_t += A_t^T . dx'   (A_t = per-type gathered source states, recomputed from the target CSR)
//          dh   += G_t . W_t^T   (G_t[s] = sum of dx'[target] over the type-t messages LEAVING s: source CSR)
//
// Kernels: elementwise cell gradients, one CSR gather for all edge types, a 64x64-tile FFMA GEMM  C (+)= sum_s A_s . B_s^T
// for the data gradients and a split-row  C_s += A_s^T . B  with fp32 atomics for the weight (+ bias) gradients; the
// segment lists keep it at ~12 launches per timestep whatever the number of edge types and residual inputs.
#pragma once
#include "ggnn_common.cuh"

namespace ggnn {
namespace bwd {

// ---------------------------------------------------------------- C[M,N] (+)= sum_s A_s[M,K] . B_s[N,K]^T
// A_s = A + s*a_stride (row stride lda), B_s = B + s*b_stride (row stride ldb): one launch covers the per-edge-type sum
// dh += sum_t G_t . W_t^T  (A = [G_0 | .. | G_{T-1}] side by side, B = the stacked [T][D][D] weights).
// 128x64 tile, 128 threads x (8x8) outputs, K in slabs of 16 through double-buffered shared memory (register-staged
// float4 global loads).  Requires K, lda, ldb, ldc, a_stride, b_stride multiples of 4 and 16-byte aligned bases
// (hidden sizes are multiples of 4 and every buffer is 16-byte aligned -- checked by the caller).
constexpr int NT_BM = 128, NT_BN = 64, GEMM_BK = 16;
template <bool ACC>
__global__ void __launch_bounds__(128) gemm_nt_kernel(const float* __restrict__ A, int lda, int a_stride, const float* __restrict__ B, int ldb,
                                                      int b_stride, int nseg, float* __restrict__ C, int ldc, int M, int N, int K) {
    __shared__ __align__(16) float As[2][GEMM_BK][NT_BM + 4];
    __shared__ __align__(16) float Bs[2][GEMM_BK][NT_BN + 4];
    const int tid = threadIdx.x, tx = tid & 7, ty = tid >> 3;
    const int m0 = blockIdx.y * NT_BM, n0 = blockIdx.x * NT_BN;
    const int kslabs = (K + GEMM_BK - 1) / GEMM_BK, nit = nseg * kslabs;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float4 ra[4], rb[2];
    auto load_global = [&](int it) {
        const int sg = it / kslabs, k0 = (it - sg * kslabs) * GEMM_BK;
        const float* Ag = A + (size_t)sg * a_stride;
        const float* Bg = B + (size_t)sg * b_stride;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int f = tid + j * 128, row = f >> 2, kq = (f & 3) * 4;
            ra[j] = (m0 + row < M && k0 + kq < K) ? *reinterpret_cast<const float4*>(Ag + (size_t)(m0 + row) * lda + k0 + kq) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int f = tid + j * 128, row = f >> 2, kq = (f & 3) * 4;
            rb[j] = (n0 + row < N && k0 + kq < K) ? *reinterpret_cast<const float4*>(Bg + (size_t)(n0 + row) * ldb + k0 + kq) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto store_shared = [&](int buf) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int f = tid + j * 128, row = f >> 2, kq = (f & 3) * 4;
            As[buf][kq + 0][row] = ra[j].x; As[buf][kq + 1][row] = ra[j].y; As[buf][kq + 2][row] = ra[j].z; As[buf][kq + 3][row] = ra[j].w;
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int f = tid + j * 128, row = f >> 2, kq = (f & 3) * 4;
            Bs[buf][kq + 0][row] = rb[j].x; Bs[buf][kq + 1][row] = rb[j].y; Bs[buf][kq + 2][row] = rb[j].z; Bs[buf][kq + 3][row] = rb[j].w;
        }
    };
    load_global(0);
    store_shared(0);
    __syncthreads();
    for (int it = 0; it < nit; ++it) {
        const int buf = it & 1;
        if (it + 1 < nit) load_global(it + 1);
#pragma unroll
        for (int kk = 0; kk < GEMM_BK; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 8]), a1 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 8 + 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]), b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][32 + tx * 4]);   // columns tx*4.. and 32+tx*4..: conflict-free
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w}, b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (it + 1 < nit) store_shared(buf ^ 1);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + ty * 8 + i;
        if (m >= M) continue;
#pragma unroll
        for (int jq = 0; jq < 2; ++jq) {
            const int n = n0 + tx * 4 + jq * 32;
            if (n >= N) continue;
            float4* c = reinterpret_cast<float4*>(C + (size_t)m * ldc + n);
            float4 v = make_float4(acc[i][jq * 4], acc[i][jq * 4 + 1], acc[i][jq * 4 + 2], acc[i][jq * 4 + 3]);
            if (ACC) { const float4 o = *c; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
            *c = v;
        }
    }
}

// ---------------------------------------------------------------- weight gradients: for every segment s
//   C[s*c_stride + k*ldc + n] += sum_m A_s[m,k] . B[m,n]      (k < K; rows m split over blockIdx.z, fp32 vector atomics)
// The segments are the pieces of the cell input row ([res.. | x | h-or-rh], each its own [V,D] array) or the per-type
// gathered source states (columns t*D.. of one [V,T*D] array): one launch per weight tensor instead of one per piece.
// bias_out (optional): bias_out[n] += sum_m B[m,n] -- the bias gradient rides along with the first segment's blocks.
// 64x64 output tile, 64 threads x (8x8), rows in slabs of 16.  a_vec = 0 selects scalar loads of A (the [V,T] in-degree table
// of the edge-bias gradient, whose row length need not be a multiple of 4); B, C, ldb, ldc, N as for gemm_nt.
constexpr int MAX_SEGS = 16;
struct SegList {
    const float* p[MAX_SEGS];
    int ld[MAX_SEGS];
};
__global__ void __launch_bounds__(64) gemm_tn_atomic_kernel(SegList segs, int kblocks, int a_vec, const float* __restrict__ B, int ldb,
                                                            float* __restrict__ C, int ldc, size_t c_stride, float* __restrict__ bias_out, int M,
                                                            int N, int K, int rows_per_split) {
    __shared__ __align__(16) float As[2][GEMM_BK][64 + 4];
    __shared__ __align__(16) float Bs[2][GEMM_BK][64 + 4];
    const int tid = threadIdx.x, tx = tid & 7, ty = tid >> 3;
    const int sg = blockIdx.y / kblocks;
    const int k0 = (blockIdx.y - sg * kblocks) * 64, n0 = blockIdx.x * 64;
    const float* __restrict__ A = segs.p[sg];
    const int lda = segs.ld[sg];
    const int mb = blockIdx.z * rows_per_split, me = min(M, mb + rows_per_split);
    const bool do_bias = bias_out != nullptr && blockIdx.y == 0;
    float acc[8][8];
    float bsum = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float4 ra[4], rb[4];
    auto load_global = [&](int m0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int f = tid + j * 64, mm = f >> 4, c4 = (f & 15) * 4;
            const bool row_ok = m0 + mm < me;
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row_ok) {
                const float* ap = A + (size_t)(m0 + mm) * lda + k0 + c4;
                if (a_vec) { if (k0 + c4 < K) a = *reinterpret_cast<const float4*>(ap); }
                else {
                    if (k0 + c4 + 0 < K) a.x = ap[0];
                    if (k0 + c4 + 1 < K) a.y = ap[1];
                    if (k0 + c4 + 2 < K) a.z = ap[2];
                    if (k0 + c4 + 3 < K) a.w = ap[3];
                }
            }
            ra[j] = a;
            rb[j] = (row_ok && n0 + c4 < N) ? *reinterpret_cast<const float4*>(B + (size_t)(m0 + mm) * ldb + n0 + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto store_shared = [&](int buf) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int f = tid + j * 64, mm = f >> 4, c4 = (f & 15) * 4;
            *reinterpret_cast<float4*>(&As[buf][mm][c4]) = ra[j];
            *reinterpret_cast<float4*>(&Bs[buf][mm][c4]) = rb[j];
        }
    };
    const int nit = (me - mb + GEMM_BK - 1) / GEMM_BK;
    if (nit > 0) {
        load_global(mb);
        store_shared(0);
    }
    __syncthreads();
    for (int it = 0; it < nit; ++it) {
        const int buf = it & 1;
        if (it + 1 < nit) load_global(mb + (it + 1) * GEMM_BK);
#pragma unroll
        for (int mm = 0; mm < GEMM_BK; ++mm) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][mm][ty * 8]), a1 = *reinterpret_cast<const float4*>(&As[buf][mm][ty * 8 + 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][mm][tx * 4]), b1 = *reinterpret_cast<const float4*>(&Bs[buf][mm][32 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w}, b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (do_bias) {
#pragma unroll
            for (int mm = 0; mm < GEMM_BK; ++mm) bsum += Bs[buf][mm][tid];
        }
        if (it + 1 < nit) store_shared(buf ^ 1);
        __syncthreads();
    }
    float* Cs = C + (size_t)sg * c_stride;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int k = k0 + ty * 8 + i;
        if (k >= K) continue;
#pragma unroll
        for (int jq = 0; jq < 2; ++jq) {
            const int n = n0 + tx * 4 + jq * 32;
            if (n >= N) continue;
            atomicAdd(reinterpret_cast<float4*>(Cs + (size_t)k * ldc + n), make_float4(acc[i][jq * 4], acc[i][jq * 4 + 1], acc[i][jq * 4 + 2], acc[i][jq * 4 + 3]));
        }
    }
    if (do_bias && n0 + tid < N) atomicAdd(bias_out + n0 + tid, bsum);
}

// ---------------------------------------------------------------- column sums: dst[n] += sum_m src[m, n]  (optionally weighted by w[m*wstride])
__global__ void __launch_bounds__(256) colsum_atomic_kernel(const float* __restrict__ src, int ld, const float* __restrict__ w, int wstride,
                                                            float* __restrict__ dst, int M, int N, int rows_per_block) {
    const int n = blockIdx.x * 256 + threadIdx.x;
    if (n >= N) return;
    const int mb = blockIdx.y * rows_per_block, me = min(M, mb + rows_per_block);
    float s = 0.f;
    for (int m = mb; m < me; ++m) s = fmaf(w ? w[(size_t)m * wstride] : 1.0f, src[(size_t)m * ld + n], s);
    atomicAdd(dst + n, s);
}

// ---------------------------------------------------------------- elementwise cell gradients
__device__ __forceinline__ float act_grad_from_output(float y, int act) { return act == ACT_TANH ? (1.0f - y * y) : (y > 0.0f ? 1.0f : 0.0f); }

// GRU part 1: dpc = dh'(1-u) act'(c) ; dpg[:, D:2D] = dh'(h-c) u(1-u) ; dh = dh' u ; rh = r h
__global__ void gru_bwd1_kernel(const float* __restrict__ dhn, const float* __restrict__ h, const float* __restrict__ r, const float* __restrict__ u,
                                const float* __restrict__ c, float* __restrict__ dpc, float* __restrict__ dpg, float* __restrict__ dh,
                                float* __restrict__ rh, long long n, int D, int act) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / D;
        const int col = (int)(i - row * D);
        const float g = dhn[i], uu = u[i], cc = c[i], hh = h[i];
        dpc[i] = g * (1.0f - uu) * act_grad_from_output(cc, act);
        dpg[row * 2 * D + D + col] = g * (hh - cc) * uu * (1.0f - uu);
        dh[i] = g * uu;
        rh[i] = r[i] * hh;
    }
}
// GRU part 2: drh = dXc[:, rh segment] ; dh += drh r ; dpg[:, 0:D] = drh h r(1-r)
__global__ void gru_bwd2_kernel(const float* __restrict__ dXc, int ldx, int rh_off, const float* __restrict__ h, const float* __restrict__ r,
                                float* __restrict__ dpg, float* __restrict__ dh, long long n, int D) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / D;
        const int col = (int)(i - row * D);
        const float drh = dXc[row * ldx + rh_off + col], rr = r[i];
        dh[i] += drh * rr;
        dpg[row * 2 * D + col] = drh * h[i] * rr * (1.0f - rr);
    }
}
// CudnnCompatibleGRUCell (sparse:105-108):  c = act(x.K_in + b_in + r*q),  q = h.K_hid + b_hid (saved by the forward)
//   dpc = dh'(1-u) act'(c)   dq = dpc r   dpg[:, 0:D] = dpc q r(1-r)   dpg[:, D:2D] = dh'(h-c) u(1-u)   dh = dh' u
__global__ void cudnn_gru_bwd1_kernel(const float* __restrict__ dhn, const float* __restrict__ h, const float* __restrict__ r, const float* __restrict__ u,
                                      const float* __restrict__ c, const float* __restrict__ q, float* __restrict__ dpc, float* __restrict__ dq,
                                      float* __restrict__ dpg, float* __restrict__ dh, long long n, int D, int act) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / D;
        const int col = (int)(i - row * D);
        const float g = dhn[i], uu = u[i], cc = c[i], hh = h[i], rr = r[i];
        const float dp = g * (1.0f - uu) * act_grad_from_output(cc, act);
        dpc[i] = dp;
        dq[i] = dp * rr;
        dpg[row * 2 * D + col] = dp * q[i] * rr * (1.0f - rr);
        dpg[row * 2 * D + D + col] = g * (hh - cc) * uu * (1.0f - uu);
        dh[i] = g * uu;
    }
}
// RNN: dpc = dh' act'(h')   (yscale = keep_prob undoes the state dropout's 1/keep on the saved output; dropped entries have dh' = 0)
__global__ void rnn_bwd1_kernel(const float* __restrict__ dhn, const float* __restrict__ hnew, float* __restrict__ dpc, long long n, int act, float yscale) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dpc[i] = dhn[i] * act_grad_from_output(hnew[i] * yscale, act);
}
// state dropout backward, in place: d(pre-dropout state) = d(state) * mask / keep   (mask regenerated, ggnn_common.cuh)
__global__ void dropout_grad_kernel(float* __restrict__ dhn, unsigned long long seed, int gstep, int V, int D, float keep, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int row = (int)(i / D), col = (int)(i - (long long)row * D);
        dhn[i] = dropout_apply(dhn[i], seed, gstep, V, D, row, col, keep);
    }
}
// Split the gradient of the cell input row [res_0 .. res_{R-1} | x | h-or-rh]:
//   dres_i[v] += dX[v, i*D..]   dxp[v] = dX[v, x segment] (/ denom)   (GRU second pass / RNN: dh (+)= dX[v, last segment])
__global__ void split_input_grad_kernel(const float* __restrict__ dXa, const float* __restrict__ dXb, int ldx, int nres,
                                        float* const* __restrict__ dres, float* __restrict__ dxp, const float* __restrict__ denom,
                                        float* __restrict__ dh, int dh_from_a, int dh_from_b, int dh_accumulate, long long n, int D) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / D;
        const int col = (int)(i - row * D);
        const float* a = dXa + row * ldx;
        const float* b = dXb ? dXb + row * ldx : nullptr;
        for (int s = 0; s < nres; ++s) dres[s][i] += a[s * D + col] + (b ? b[s * D + col] : 0.0f);
        float x = a[nres * D + col] + (b ? b[nres * D + col] : 0.0f);
        if (denom) x = x / denom[row];
        dxp[i] = x;
        float hg = 0.0f;
        if (dh_from_a) hg += a[(nres + 1) * D + col];
        if (dh_from_b && b) hg += b[(nres + 1) * D + col];
        if (dh_from_a || dh_from_b) dh[i] = dh_accumulate ? dh[i] + hg : hg;
    }
}
__global__ void add_inplace_kernel(float* __restrict__ dst, const float* __restrict__ src, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dst[i] += src[i];
}

// ---------------------------------------------------------------- gathers, all edge types in one launch (one warp per node):
//   out[v, t*D + :] = sum_{slots of row (v*T+t)} in[idx[slot], :]        out is [V, T*D]
// blockIdx.y = 0: A_t from the target-keyed CSR over the states; 1: G_t from the source-keyed CSR over dx'.
// w (optional): per-slot weight (the attention probability), looked up as w[widx ? widx[slot] : slot]
struct GatherJob { const int* row_ptr; const int* idx; const float* in; float* out; const float* w; const int* widx; };
__global__ void __launch_bounds__(256) csr_gather_all_kernel(GatherJob j0, GatherJob j1, int V, int D, int T) {
    const GatherJob jb = blockIdx.y == 0 ? j0 : j1;
    const int v = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (v >= V) return;
    for (int t = 0; t < T; ++t) {
        const int beg = jb.row_ptr[(size_t)v * T + t], end = jb.row_ptr[(size_t)v * T + t + 1];
        float* o = jb.out + ((size_t)v * T + t) * D;
        for (int c4 = lane; c4 < (D >> 2); c4 += 32) {
            float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
            if (jb.w) {
                for (int m = beg; m < end; ++m) {
                    const float a = jb.w[jb.widx ? jb.widx[m] : m];
                    const float4 x = *reinterpret_cast<const float4*>(jb.in + (size_t)jb.idx[m] * D + (c4 << 2));
                    s.x = fmaf(a, x.x, s.x); s.y = fmaf(a, x.y, s.y); s.z = fmaf(a, x.z, s.z); s.w = fmaf(a, x.w, s.w);
                }
            } else {
                for (int m = beg; m < end; ++m) {
                    const float4 x = *reinterpret_cast<const float4*>(jb.in + (size_t)jb.idx[m] * D + (c4 << 2));
                    s.x += x.x; s.y += x.y; s.z += x.z; s.w += x.w;
                }
            }
            *reinterpret_cast<float4*>(o + (c4 << 2)) = s;
        }
    }
}

// ---------------------------------------------------------------- propagation attention backward (sparse:170-196)
// incoming[v] = sum_m alpha_m (h[src_m] W_t),  alpha = softmax over the messages into v of  s_m = a_t <h[src_m], h[v]>  (+1e-7 in the
// denominator).  With P = dx' . W^T ([V, T*D], one GEMM):  d alpha_m = <P[v, t*D..], h[src_m]>,
//   d s_m = alpha_m (d alpha_m - sum_k alpha_k d alpha_k),   d a_t += d s_m <h[src], h[v]>,
//   d h[v] += sum_m d s_m a_t h[src_m]   (this kernel, one warp per target),   d h[src] += d s_m a_t h[v]  (source kernel below).
// dsa[slot] = d s_m a_t is left for the source kernel; scratch[slot] holds d alpha in between.
// DET (the deterministic backward): instead of atomics into d_att_w, every block writes its per-type sums, added over its 8 warps in
// warp order, to daw_part[block][T]; a fixed-order column sum (ggnn_bwd_tc.cuh) adds them to d_att_w.
template <bool DET>
__global__ void __launch_bounds__(256) attention_bwd_target_kernel(const int* __restrict__ row_ptr, const int* __restrict__ csr_src,
                                                                   const float* __restrict__ h, const float* __restrict__ P,
                                                                   const float* __restrict__ alpha, const float* __restrict__ att_w,
                                                                   float* __restrict__ dsa, float* __restrict__ dh, float* __restrict__ d_att_w,
                                                                   int V, int D, int T, float* __restrict__ daw_part) {
    __shared__ float s_daw[16];
    __shared__ float s_dawp[DET ? 8 : 1][16];
    if (threadIdx.x < 16) s_daw[threadIdx.x] = 0.f;
    if (DET && threadIdx.x < 8 * 16) s_dawp[threadIdx.x >> 4][threadIdx.x & 15] = 0.f;
    __syncthreads();
    const int v = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (v < V) {
        const float* hv = h + (size_t)v * D;
        float acc = 0.f;   // sum_k alpha_k d alpha_k
        for (int t = 0; t < T; ++t) {
            const float* Pv = P + ((size_t)v * T + t) * D;
            for (int m = row_ptr[(size_t)v * T + t]; m < row_ptr[(size_t)v * T + t + 1]; ++m) {
                const float* hs = h + (size_t)csr_src[m] * D;
                float dal = 0.f;
                for (int c = lane; c < D; c += 32) dal = fmaf(Pv[c], hs[c], dal);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) dal += __shfl_xor_sync(0xffffffffu, dal, o);
                if (lane == 0) dsa[m] = dal;
                acc = fmaf(alpha[m], dal, acc);
            }
        }
        __syncwarp();
        float dhv[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) dhv[j] = 0.f;
        for (int t = 0; t < T; ++t) {
            const float aw = att_w[t];
            float daw = 0.f;
            for (int m = row_ptr[(size_t)v * T + t]; m < row_ptr[(size_t)v * T + t + 1]; ++m) {
                const float* hs = h + (size_t)csr_src[m] * D;
                const float ds = alpha[m] * (dsa[m] - acc);
                float dot = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = lane + 32 * j;
                    if (c < D) { const float x = hs[c]; dot = fmaf(x, hv[c], dot); dhv[j] = fmaf(ds * aw, x, dhv[j]); }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
                daw = fmaf(ds, dot, daw);
                __syncwarp();
                if (lane == 0) dsa[m] = ds * aw;
            }
            if (DET) { if (lane == 0) s_dawp[threadIdx.x >> 5][t] = daw; }
            else if (lane == 0 && d_att_w && daw != 0.f) atomicAdd(&s_daw[t], daw);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = lane + 32 * j;
            if (c < D) dh[(size_t)v * D + c] += dhv[j];
        }
    }
    __syncthreads();
    if (DET) {
        if (daw_part && threadIdx.x < T) {
            float s = 0.f;
            for (int w = 0; w < 8; ++w) s += s_dawp[w][threadIdx.x];
            daw_part[(size_t)blockIdx.x * T + threadIdx.x] = s;
        }
    } else if (d_att_w && threadIdx.x < T && s_daw[threadIdx.x] != 0.f) atomicAdd(d_att_w + threadIdx.x, s_daw[threadIdx.x]);
}
// d h[s] += sum over the messages LEAVING s of dsa[target-CSR slot] * h[target]     (source-keyed CSR, one warp per source)
__global__ void __launch_bounds__(256) attention_bwd_source_kernel(const int* __restrict__ trow, const int* __restrict__ ttgt,
                                                                   const int* __restrict__ tslot, const float* __restrict__ h,
                                                                   const float* __restrict__ dsa, float* __restrict__ dh, int V, int D, int T) {
    const int s = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (s >= V) return;
    const int beg = trow[(size_t)s * T], end = trow[(size_t)(s + 1) * T];
    if (beg == end) return;
    for (int c4 = lane; c4 < (D >> 2); c4 += 32) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = beg; j < end; ++j) {
            const float w = dsa[tslot[j]];
            const float4 x = *reinterpret_cast<const float4*>(h + (size_t)ttgt[j] * D + (c4 << 2));
            a.x = fmaf(w, x.x, a.x); a.y = fmaf(w, x.y, a.y); a.z = fmaf(w, x.z, a.z); a.w = fmaf(w, x.w, a.w);
        }
        float4* o = reinterpret_cast<float4*>(dh + (size_t)s * D + (c4 << 2));
        float4 cur = *o;
        cur.x += a.x; cur.y += a.y; cur.z += a.z; cur.w += a.w;
        *o = cur;
    }
}
// dense adjacency [b][T][v][v]: out[g*nv+i] = sum_j A[g,t,i,j] in[g*nv+j]   (transpose: sum_j A[g,t,j,i] in[g*nv+j])
__global__ void __launch_bounds__(256) dense_gather_sum_kernel(const float* __restrict__ adj, const float* __restrict__ in, float* __restrict__ out,
                                                               int ldo, int V, int D, int T, int t, int nv, int transpose) {
    const int v = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (v >= V) return;
    const int g = v / nv, i = v - g * nv;
    const float* base = adj + ((size_t)g * T + t) * nv * nv;
    for (int c4 = lane; c4 < (D >> 2); c4 += 32) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = 0; j < nv; ++j) {
            const float a = transpose ? base[(size_t)j * nv + i] : base[(size_t)i * nv + j];
            if (a != 0.0f) {
                const float4 x = *reinterpret_cast<const float4*>(in + (size_t)(g * nv + j) * D + (c4 << 2));
                s.x = fmaf(a, x.x, s.x); s.y = fmaf(a, x.y, s.y); s.z = fmaf(a, x.z, s.z); s.w = fmaf(a, x.w, s.w);
            }
        }
        *reinterpret_cast<float4*>(out + (size_t)v * ldo + (c4 << 2)) = s;
    }
}

}  // namespace bwd
}  // namespace ggnn
