// V x V attention stages for LARGE graphs (V > 32): the 1-D adaptive graph convolution of the IMU / late-fusion models
// (torch_src/models/mmargcn/graph_convolution.py:56-113, AGCNGraphConvolution; :12-53, STGCNGraphConvolution; SURVEY 8 f2), whose
// graphs have T * signals nodes (up to 652), so the per-sample V x V matrices (1.7 MB each) no longer fit the shared-memory-resident
// kernels of joint.cu / mix_tc.cu.  Every product of that operator is a small batched GEMM over the node axis:
//     score   S_k  = theta_k^T phi_k          gram        A(u, c) K-contiguous,  B(c, v) K-contiguous
//     mix     Z_k  = X . G_k                  AGG_FWD     A(v, u) = G[u][v] M-contiguous,  B(u, c) N-contiguous
//     dX     += dZ_k . G_k^T                  AGG_BWD     A(u, v) K-contiguous,  B(v, c) N-contiguous, summed over k (segments)
//     dtheta  = dS_k . phi_k,  dphi = dS_k^T theta_k       (both forms again)
//     STGCN   out = support . adj^T           one fixed matrix for the whole batch (batch stride 0)
// so ONE strided, batched, segmented fp32 FFMA GEMM (64 x 64 tiles, 4 x 4 register blocks, operands staged through shared memory along
// whichever of their two axes is contiguous) serves all of them, exact fp32 like the FFMA kernels of the small-V path.
// The column softmax and its backward walk the V x V matrices with one warp per column.
#include "common.cuh"

namespace agcn {

struct BigGemm {
    const float* a; const float* b; float* c;
    int batch2, segs, m, n, k;
    long long a_b1, a_b2, a_seg, a_m, a_k;
    long long b_b1, b_b2, b_seg, b_k, b_n;
    long long c_b1, c_b2, c_m;          // c_n = 1
    float alpha;
    int accumulate;
};

constexpr int kBM = 64, kBN = 64, kBK = 16;

// C[b][m][n] (+)= alpha * sum_seg sum_k A[b][seg](m, k) * B[b][seg](k, n);  grid = (n tiles, m tiles, batch1 * batch2)
__global__ void __launch_bounds__(256) big_gemm_kernel(BigGemm p) {
    __shared__ float as[kBK][kBM + 4];
    __shared__ float bs[kBK][kBN + 4];
    const int b1 = blockIdx.z / p.batch2, b2 = blockIdx.z - b1 * p.batch2;
    const int m0 = blockIdx.y * kBM, n0 = blockIdx.x * kBN;
    const float* abase = p.a + b1 * p.a_b1 + b2 * p.a_b2;
    const float* bbase = p.b + b1 * p.b_b1 + b2 * p.b_b2;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // 16 x 16 threads, each a 4 x 4 block of the tile
    float acc[4][4] = {};
    // loader mappings: consecutive threads walk the CONTIGUOUS axis of the operand
    const bool a_kc = p.a_k == 1, b_nc = p.b_n == 1;
    for (int seg = 0; seg < p.segs; ++seg) {
        const float* ap = abase + seg * p.a_seg;
        const float* bp = bbase + seg * p.b_seg;
        for (int k0 = 0; k0 < p.k; k0 += kBK) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int e = threadIdx.x + i * 256;              // 1024 elements per operand tile
                int mm, kk;
                if (a_kc) { kk = e & (kBK - 1); mm = e >> 4; } else { mm = e & (kBM - 1); kk = e >> 6; }
                const int gm = m0 + mm, gk = k0 + kk;
                as[kk][mm] = (gm < p.m && gk < p.k) ? __ldg(ap + gm * p.a_m + gk * p.a_k) : 0.f;
                int nn, kb;
                if (b_nc) { nn = e & (kBN - 1); kb = e >> 6; } else { kb = e & (kBK - 1); nn = e >> 4; }
                const int gn = n0 + nn, gkb = k0 + kb;
                bs[kb][nn] = (gn < p.n && gkb < p.k) ? __ldg(bp + gkb * p.b_k + gn * p.b_n) : 0.f;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < kBK; ++kk) {
                const float4 av = *reinterpret_cast<const float4*>(&as[kk][ty * 4]);
                const float4 bv = *reinterpret_cast<const float4*>(&bs[kk][tx * 4]);
                const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
            }
            __syncthreads();
        }
    }
    float* cbase = p.c + b1 * p.c_b1 + b2 * p.c_b2;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= p.m) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= p.n) continue;
            float* dst = cbase + gm * p.c_m + gn;
            const float v = p.alpha * acc[i][j];
            *dst = p.accumulate ? *dst + v : v;
        }
    }
}

static int launch_big_gemm(const BigGemm& p, int batch1, cudaStream_t s, const char* what) {
    AGCN_REQUIRE((p.a_k == 1 || p.a_m == 1) && (p.b_n == 1 || p.b_k == 1), AGCN_ERR_UNSUPPORTED,
                 "%s: each operand needs a unit stride along one of its axes", what);
    dim3 grid((unsigned)ceil_div(p.n, kBN), (unsigned)ceil_div(p.m, kBM), (unsigned)(batch1 * p.batch2));
    AGCN_REQUIRE(grid.z <= 65535u && grid.y <= 65535u, AGCN_ERR_UNSUPPORTED, "%s: batch too large for one launch", what);
    big_gemm_kernel<<<grid, 256, 0, s>>>(p);
    return check_launch(what);
}

// p[n][k][:, v] = softmax_u(scale * s[n][k][u][v]);  g = p + adj_a[k] + adj_b[k].   One warp per 32 columns: lane = column.
__global__ void __launch_bounds__(256) big_attention_fwd_kernel(const float* s, const float* adj_a, const float* adj_b, float* p, float* g,
                                                                int groups, int v, float scale) {
    const int nk = blockIdx.y, k = nk % groups;
    const int col = blockIdx.x * 256 + threadIdx.x;
    if (col >= v) return;
    const float* sp = s + (long long)nk * v * v + col;
    float mx = -INFINITY;
    for (int u = 0; u < v; ++u) mx = fmaxf(mx, sp[(long long)u * v] * scale);
    float sum = 0.f;
    for (int u = 0; u < v; ++u) sum += expf(sp[(long long)u * v] * scale - mx);
    const float inv = 1.f / sum;
    const float* aa = adj_a + (long long)k * v * v + col;
    const float* ab = adj_b + (long long)k * v * v + col;
    float* pp = p + (long long)nk * v * v + col;
    float* gp = g + (long long)nk * v * v + col;
    for (int u = 0; u < v; ++u) {
        const float pv = expf(sp[(long long)u * v] * scale - mx) * inv;
        pp[(long long)u * v] = pv;
        gp[(long long)u * v] = pv + aa[(long long)u * v] + ab[(long long)u * v];
    }
}

// ds = scale * p * (dG - colsum_u(p * dG))   (dg_sum: the summed dG, here simply dg_part with one chunk)
__global__ void __launch_bounds__(256) big_attention_bwd_kernel(const float* dg, const float* p, float* dg_sum, float* ds, int v, float scale) {
    const int nk = blockIdx.y;
    const int col = blockIdx.x * 256 + threadIdx.x;
    if (col >= v) return;
    const long long base = (long long)nk * v * v + col;
    float dot = 0.f;
    for (int u = 0; u < v; ++u) dot = fmaf(p[base + (long long)u * v], dg[base + (long long)u * v], dot);
    for (int u = 0; u < v; ++u) {
        const float d = dg[base + (long long)u * v];
        dg_sum[base + (long long)u * v] = d;
        ds[base + (long long)u * v] = scale * p[base + (long long)u * v] * (d - dot);
    }
}

__global__ void big_sum_over_samples_kernel(const float* dg, float* dadj_b, int nb, long long per_sample) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= per_sample) return;
    float s = 0.f;
    for (int n = 0; n < nb; ++n) s += dg[n * per_sample + i];
    dadj_b[i] = s;
}

}  // namespace agcn

using namespace agcn;

// ---- internal entry points used by joint.cu when V exceeds the shared-memory-resident kernels
int agcn_joint_gram_big(const float* a, const float* b, float* out, int nb, int t, int v, int lda, int ldb, int groups,
                        int offa, int stridea, int offb, int strideb, int width, void* stream) {
    // out[n][0][g][u][v] = sum_t sum_c a[n][t][u][offa + g*stridea + c] * b[n][t][v][offb + g*strideb + c]: segments = timesteps
    BigGemm p{};
    p.a = a + offa; p.b = b + offb; p.c = out;
    p.batch2 = groups; p.segs = t; p.m = v; p.n = v; p.k = width;
    p.a_b1 = (long long)t * v * lda; p.a_b2 = stridea; p.a_seg = (long long)v * lda; p.a_m = lda; p.a_k = 1;
    p.b_b1 = (long long)t * v * ldb; p.b_b2 = strideb; p.b_seg = (long long)v * ldb; p.b_k = 1; p.b_n = ldb;
    p.c_b1 = (long long)groups * v * v; p.c_b2 = (long long)v * v; p.c_m = v;
    p.alpha = 1.f; p.accumulate = 0;
    return launch_big_gemm(p, nb, static_cast<cudaStream_t>(stream), "agcn_joint_gram(big V)");
}

int agcn_attention_fwd_big(const float* s_part, const float* adj_a, const float* adj_b, float* p, float* g,
                           int nb, int groups, int v, float scale, void* stream) {
    dim3 grid((unsigned)ceil_div(v, 256), (unsigned)(nb * groups));
    big_attention_fwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(s_part, adj_a, adj_b, p, g, groups, v, scale);
    return check_launch("agcn_attention_fwd(big V)");
}

int agcn_attention_bwd_big(const float* dg_part, const float* p, float* dg_sum, float* ds, float* dadj_b,
                           int nb, int groups, int v, float scale, void* stream) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    dim3 grid((unsigned)ceil_div(v, 256), (unsigned)(nb * groups));
    big_attention_bwd_kernel<<<grid, 256, 0, s>>>(dg_part, p, dg_sum, ds, v, scale);
    int rc = check_launch("agcn_attention_bwd(big V)");
    if (rc) return rc;
    const long long per = (long long)groups * v * v;
    big_sum_over_samples_kernel<<<ceil_div(per, 256), 256, 0, s>>>(dg_sum, dadj_b, nb, per);
    return check_launch("agcn_attention_bwd(big V, dadj_b)");
}

int agcn_joint_mix_big(const float* in, const float* mats, float* out, int nb, int t, int v, int ldin, int ldout, int width,
                       int mode, int accumulate, void* stream) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    BigGemm p{};
    p.alpha = 1.f;
    const long long mat = (long long)v * v;
    if (mode == AGCN_MIX_AGG_FWD) {
        // out[n][t][v][k*W + c] (+)= sum_u G[n][k][u][v] * in[n][t][u][c]: batch (n*t, k), A(m = v, k = u) = G[u][v]
        p.a = mats; p.b = in; p.c = out;
        p.batch2 = 3; p.segs = 1; p.m = v; p.n = width; p.k = v;
        p.a_b1 = 0; p.a_b2 = mat; p.a_m = 1; p.a_k = v;
        p.b_b1 = (long long)v * ldin; p.b_b2 = 0; p.b_k = ldin; p.b_n = 1;
        p.c_b1 = (long long)v * ldout; p.c_b2 = width; p.c_m = ldout;
        p.accumulate = accumulate;
        // batch1 runs over (n, t): the matrix stride follows n only -> one launch per sample block of timesteps
        for (int n = 0; n < nb; ++n) {
            BigGemm q = p;
            q.a = mats + (long long)n * 3 * mat;
            q.b = in + (long long)n * t * v * ldin;
            q.c = out + (long long)n * t * v * ldout;
            int rc = launch_big_gemm(q, t, s, "agcn_joint_mix(big V, aggregate)");
            if (rc) return rc;
        }
        return AGCN_OK;
    }
    if (mode == AGCN_MIX_AGG_BWD) {
        // out[n][t][u][c] (+)= sum_k sum_v G[n][k][u][v] * in[n][t][v][k*W + c]: segments = subsets
        p.batch2 = 1; p.segs = 3; p.m = v; p.n = width; p.k = v;
        p.a_seg = mat; p.a_m = v; p.a_k = 1;
        p.b_b1 = (long long)v * ldin; p.b_seg = width; p.b_k = ldin; p.b_n = 1;
        p.c_b1 = (long long)v * ldout; p.c_m = ldout;
        p.accumulate = accumulate;
        for (int n = 0; n < nb; ++n) {
            BigGemm q = p;
            q.a = mats + (long long)n * 3 * mat;
            q.b = in + (long long)n * t * v * ldin;
            q.c = out + (long long)n * t * v * ldout;
            int rc = launch_big_gemm(q, t, s, "agcn_joint_mix(big V, aggregate bwd)");
            if (rc) return rc;
        }
        return AGCN_OK;
    }
    // SCORE_BWD: in = [theta_0 phi_0 theta_1 phi_1 theta_2 phi_2], mats = dS
    //   out[.., u, theta_k c] (+)= sum_v dS[k][u][v] * in[.., v, phi_k c];   out[.., v, phi_k c] (+)= sum_u dS[k][u][v] * in[.., u, theta_k c]
    // the theta and phi slots are disjoint columns, so each of the two GEMMs adds into its own slot
    for (int n = 0; n < nb; ++n) {
        BigGemm q{};
        q.alpha = 1.f; q.accumulate = accumulate;
        q.batch2 = 3; q.segs = 1; q.m = v; q.n = width; q.k = v;
        q.b_b1 = (long long)v * ldin; q.b_b2 = 2 * width; q.b_k = ldin; q.b_n = 1;
        q.c_b1 = (long long)v * ldout; q.c_b2 = 2 * width; q.c_m = ldout;
        q.a = mats + (long long)n * 3 * mat; q.a_b1 = 0; q.a_b2 = mat;
        // d theta: A(m = u, k = v) = dS[u][v], B = phi (channel offset W), C = theta slot (offset 0)
        q.a_m = v; q.a_k = 1;
        q.b = in + (long long)n * t * v * ldin + width;
        q.c = out + (long long)n * t * v * ldout;
        int rc = launch_big_gemm(q, t, s, "agcn_joint_mix(big V, d theta)");
        if (rc) return rc;
        // d phi: A(m = v, k = u) = dS[u][v], B = theta (offset 0), C = phi slot (offset W)
        q.a_m = 1; q.a_k = v;
        q.b = in + (long long)n * t * v * ldin;
        q.c = out + (long long)n * t * v * ldout + width;
        rc = launch_big_gemm(q, t, s, "agcn_joint_mix(big V, d phi)");
        if (rc) return rc;
    }
    return AGCN_OK;
}

/* out[b][v][c] (+)= sum_u mat[v][u] * in[b][u][c]  (transpose_mat == 0)   or   sum_u mat[u][v] * in[b][u][c]  (transpose_mat != 0)
 * One fixed matrix for the whole batch: the STGCN graph convolution support . adj^T (graph_convolution.py:45) and its input gradient. */
extern "C" AGCN_API int agcn_node_mix(const float* in, const float* mat, float* out, int batch, int v, int channels,
                                      int transpose_mat, int accumulate, void* stream) {
    AGCN_REQUIRE(in && mat && out, AGCN_ERR_NULL, "agcn_node_mix: null pointer");
    AGCN_REQUIRE(batch > 0 && v > 0 && channels > 0, AGCN_ERR_BAD_SHAPE, "agcn_node_mix: bad shape");
    BigGemm p{};
    p.a = mat; p.b = in; p.c = out;
    p.batch2 = 1; p.segs = 1; p.m = v; p.n = channels; p.k = v;
    if (transpose_mat) { p.a_m = 1; p.a_k = v; } else { p.a_m = v; p.a_k = 1; }
    p.b_b1 = (long long)v * channels; p.b_k = channels; p.b_n = 1;
    p.c_b1 = (long long)v * channels; p.c_m = channels;
    p.alpha = 1.f; p.accumulate = accumulate;
    return launch_big_gemm(p, batch, static_cast<cudaStream_t>(stream), "agcn_node_mix");
}
