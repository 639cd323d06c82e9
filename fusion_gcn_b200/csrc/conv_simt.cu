// FP32 FFMA implicit-GEMM kernels (parity mode + fallback for shapes the tcgen05 path does not take):
//   agcn_conv_fwd   : y[rows][cout] (+)= bias + sum_tap x[gather(row,tap)][cin] . w[cout][tap][cin]
//   agcn_conv_wgrad : dw[cout][tap][cin] = sum_rows dy[row][cout] * x[gather(row,tap)][cin]
// Channels-last activations, rows = (nb, t, v).  Reference arithmetic: nn.Conv2d at
// torch_src/models/mmargcn/agcn.py:41-42,71-73,77 and its autograd backward.
#include "common.cuh"
#include <stdlib.h>

namespace agcn {

struct ConvArgs {
    const float* x; const float* w; const float* bias; float* y;
    int nb, t_in, t_out, v, cin, cout, taps, stride, pad, transposed, accumulate;
    long long rows_out;
    PostOp post;           // eval-mode fused tail (all NULL / 0: plain convolution)
};

__device__ __forceinline__ int gather_t(int to, int tap, const ConvArgs& a) {
    // returns input time index or -1
    if (!a.transposed) {
        int ti = a.stride * to + tap - a.pad;
        return (ti >= 0 && ti < a.t_in) ? ti : -1;
    }
    int num = to + a.pad - tap;
    if (num < 0) return -1;
    if (a.stride != 1) {
        if (num % a.stride) return -1;
        num /= a.stride;
    }
    return num < a.t_in ? num : -1;
}

// 128 x 64 output tile, K step 16, 256 threads, 8x4 outputs per thread, register-prefetch double buffering.
template <bool VEC>
__global__ void __launch_bounds__(256) conv_fwd_kernel(ConvArgs a) {
    constexpr int BM = 128, BN = 64, BK = 16, LDA = BM + 4, LDB = BN + 4;
    __shared__ __align__(16) float As[2][BK][LDA];
    __shared__ __align__(16) float Bs[2][BK][LDB];
    const int tid = threadIdx.x;
    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int lrow = tid >> 2, lkq = tid & 3;

    int rn[2], rt[2], rv[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        long long r = m0 + lrow + i * 64;
        if (r < a.rows_out) {
            rv[i] = (int)(r % a.v);
            long long q = r / a.v;
            rt[i] = (int)(q % a.t_out);
            rn[i] = (int)(q / a.t_out);
        } else {
            rn[i] = -1; rt[i] = 0; rv[i] = 0;
        }
    }
    const int wcol = n0 + lrow;          // weight row (output channel) this thread loads
    const int kchunks = (a.cin + BK - 1) / BK;
    const int total = a.taps * kchunks;

    float ra[2][4], rb[4];
    auto load_global = [&](int it) {
        const int tap = it / kchunks;
        const int k0 = (it - tap * kchunks) * BK + lkq * 4;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            ra[i][0] = ra[i][1] = ra[i][2] = ra[i][3] = 0.f;
            if (rn[i] >= 0) {
                int ti = gather_t(rt[i], tap, a);
                if (ti >= 0) {
                    const float* p = a.x + (((long long)rn[i] * a.t_in + ti) * a.v + rv[i]) * a.cin + k0;
                    if (VEC) {
                        if (k0 < a.cin) {
                            float4 q = __ldg(reinterpret_cast<const float4*>(p));
                            ra[i][0] = q.x; ra[i][1] = q.y; ra[i][2] = q.z; ra[i][3] = q.w;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (k0 + j < a.cin) ra[i][j] = __ldg(p + j);
                    }
                }
            }
        }
        rb[0] = rb[1] = rb[2] = rb[3] = 0.f;
        if (wcol < a.cout) {
            const float* p = a.w + ((long long)wcol * a.taps + tap) * a.cin + k0;
            if (VEC) {
                if (k0 < a.cin) {
                    float4 q = __ldg(reinterpret_cast<const float4*>(p));
                    rb[0] = q.x; rb[1] = q.y; rb[2] = q.z; rb[3] = q.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) if (k0 + j < a.cin) rb[j] = __ldg(p + j);
            }
        }
    };
    auto store_smem = [&](int buf) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            As[buf][lkq * 4 + j][lrow] = ra[0][j];
            As[buf][lkq * 4 + j][lrow + 64] = ra[1][j];
            Bs[buf][lkq * 4 + j][lrow] = rb[j];
        }
    };

    const int tx = tid & 15, ty = tid >> 4;
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    load_global(0);
    store_smem(0);
    __syncthreads();
    for (int it = 0; it < total; ++it) {
        const int buf = it & 1;
        if (it + 1 < total) load_global(it + 1);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8]);
            float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8 + 4]);
            float4 b = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (it + 1 < total) store_smem(buf ^ 1);
        __syncthreads();
    }

    const int col = n0 + tx * 4;
    float bias[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.bias) {
#pragma unroll
        for (int j = 0; j < 4; ++j) if (col + j < a.cout) bias[j] = __ldg(a.bias + col + j);
    }
    const bool vec_out = ((a.cout & 3) == 0) && (col + 3 < a.cout);
    float psc[4] = {1.f, 1.f, 1.f, 1.f}, psh[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.post.scale) {
#pragma unroll
        for (int j = 0; j < 4; ++j) if (col + j < a.cout) { psc[j] = __ldg(a.post.scale + col + j); psh[j] = __ldg(a.post.shift + col + j); }
    }
    const bool has_post = a.post.scale != nullptr || a.post.res != nullptr || a.post.relu != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        long long r = m0 + ty * 8 + i;
        if (r >= a.rows_out) continue;
        float* p = a.y + r * a.cout + col;
        if (has_post) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (col + j < a.cout) {
                    float o = fmaf(acc[i][j] + bias[j], psc[j], psh[j]);
                    if (a.post.res) o += __ldg(a.post.res + r * a.cout + col + j);
                    if (a.post.relu) o = fmaxf(o, 0.f);
                    p[j] = o;
                }
            }
            continue;
        }
        if (vec_out) {
            float4 o = make_float4(acc[i][0] + bias[0], acc[i][1] + bias[1], acc[i][2] + bias[2], acc[i][3] + bias[3]);
            if (a.accumulate) {
                float4 old = *reinterpret_cast<const float4*>(p);
                o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
            }
            *reinterpret_cast<float4*>(p) = o;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (col + j < a.cout) {
                    float o = acc[i][j] + bias[j];
                    if (a.accumulate) o += p[j];
                    p[j] = o;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------ wgrad
struct WgradArgs {
    const float* dy; const float* x; float* ws_w; float* ws_b;
    int nb, t_in, t_out, v, cin, cout, taps, stride, pad;
    long long rows_out, rows_per_split;
    int ntiles, ktiles;
};

// one CTA: 64 (cout) x 64 (cin) tile of one tap, over one row split; thread tile 4x4.
template <bool VEC>
__global__ void __launch_bounds__(256) conv_wgrad_kernel(WgradArgs a) {
    constexpr int BR = 32, TN = 64, TK = 64, LD = 68;
    __shared__ __align__(16) float Ds[BR][LD];
    __shared__ __align__(16) float Xs[BR][LD];
    const int tid = threadIdx.x;
    int tile = blockIdx.x;
    const int tap = tile % a.taps; tile /= a.taps;
    const int ktile = tile % a.ktiles;
    const int ntile = tile / a.ktiles;
    const int n0 = ntile * TN, k0 = ktile * TK;
    const int split = blockIdx.y;
    const long long r_begin = (long long)split * a.rows_per_split;
    long long r_end = r_begin + a.rows_per_split;
    if (r_end > a.rows_out) r_end = a.rows_out;

    const int lr = tid >> 4, lc = (tid & 15) * 4;
    const int tx = tid & 15, ty = tid >> 4;
    const bool do_bias = (a.ws_b != nullptr) && ktile == 0 && tap == 0 && tid < TN;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float bsum = 0.f;

    for (long long rb = r_begin; rb < r_end; rb += BR) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int rr = lr + h * 16;
            const long long r = rb + rr;
            float d[4] = {0.f, 0.f, 0.f, 0.f}, xv[4] = {0.f, 0.f, 0.f, 0.f};
            if (r < r_end) {
                const float* pd = a.dy + r * a.cout + n0 + lc;
                if (VEC) {
                    if (n0 + lc < a.cout) {
                        float4 q = __ldg(reinterpret_cast<const float4*>(pd));
                        d[0] = q.x; d[1] = q.y; d[2] = q.z; d[3] = q.w;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) if (n0 + lc + j < a.cout) d[j] = __ldg(pd + j);
                }
                const int vv = (int)(r % a.v);
                const long long q2 = r / a.v;
                const int to = (int)(q2 % a.t_out);
                const int n = (int)(q2 / a.t_out);
                const int ti = a.stride * to + tap - a.pad;
                if (ti >= 0 && ti < a.t_in) {
                    const float* px = a.x + (((long long)n * a.t_in + ti) * a.v + vv) * a.cin + k0 + lc;
                    if (VEC) {
                        if (k0 + lc < a.cin) {
                            float4 q = __ldg(reinterpret_cast<const float4*>(px));
                            xv[0] = q.x; xv[1] = q.y; xv[2] = q.z; xv[3] = q.w;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (k0 + lc + j < a.cin) xv[j] = __ldg(px + j);
                    }
                }
            }
            *reinterpret_cast<float4*>(&Ds[rr][lc]) = make_float4(d[0], d[1], d[2], d[3]);
            *reinterpret_cast<float4*>(&Xs[rr][lc]) = make_float4(xv[0], xv[1], xv[2], xv[3]);
        }
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < BR; ++r) {
            float4 d4 = *reinterpret_cast<const float4*>(&Ds[r][ty * 4]);
            float4 x4 = *reinterpret_cast<const float4*>(&Xs[r][tx * 4]);
            const float dv[4] = {d4.x, d4.y, d4.z, d4.w};
            const float xw[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], xw[j], acc[i][j]);
        }
        if (do_bias) {
#pragma unroll 8
            for (int r = 0; r < BR; ++r) bsum += Ds[r][tid];
        }
        __syncthreads();
    }
    const long long wsize = (long long)a.cout * a.taps * a.cin;
    float* out = a.ws_w + (long long)split * wsize;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= a.cout) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx * 4 + j;
            if (k < a.cin) out[((long long)n * a.taps + tap) * a.cin + k] = acc[i][j];
        }
    }
    if (do_bias && n0 + tid < a.cout) a.ws_b[(long long)split * a.cout + n0 + tid] = bsum;
}

__global__ void wgrad_reduce_kernel(const float* ws_w, const float* ws_b, float* dw, float* db,
                                    long long wsize, int cout, int splits) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < wsize) {
        float s = 0.f;
        for (int k = 0; k < splits; ++k) s += ws_w[(long long)k * wsize + i];
        dw[i] = s;
    } else if (db != nullptr && i < wsize + cout) {
        long long c = i - wsize;
        float s = 0.f;
        for (int k = 0; k < splits; ++k) s += ws_b[(long long)k * cout + c];
        db[c] = s;
    }
}

// ------------------------------------------------------------------------------------------ skinny shapes (first unit)
// The first unit has 2..9 input channels (C = 3 joints coordinates, 9 after aggregation): a 64-wide GEMM tile would waste
// >90 % of its FMAs there, and these contractions are plain HBM streams.  Two dedicated kernels:
//   conv_skinny_out_kernel : y[row][co] (+)= bias + sum_ci x[row][ci] w[co][ci],  cout <= 16, cin % 4 == 0   (input gradients)
//   wgrad_skinny_kernel    : part[b][co][ci] = sum_{rows of b} dy[row][co] x[row][ci],  cin <= 16            (weight gradients)
constexpr int kSkinnyRows = 128;

__global__ void __launch_bounds__(256) conv_skinny_out_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                              const float* __restrict__ bias, float* __restrict__ y,
                                                              long long rows, int cin, int cout, int accumulate) {
    extern __shared__ __align__(16) float sm[];
    const int ld = cin + 4;
    float* xs = sm;                                   // [128][ld]
    float* ws = xs + kSkinnyRows * ld;                // [cout][cin]
    float* os = ws + cout * cin;                      // [128][cout]
    const int tid = threadIdx.x;
    for (int i = tid; i < cout * cin; i += 256) ws[i] = __ldg(w + i);
    const int cq = cin >> 2;
    for (long long r0 = (long long)blockIdx.x * kSkinnyRows; r0 < rows; r0 += (long long)gridDim.x * kSkinnyRows) {
        const int rn = (rows - r0) < kSkinnyRows ? (int)(rows - r0) : kSkinnyRows;
        __syncthreads();
        const float4* src = reinterpret_cast<const float4*>(x + r0 * cin);
        for (int i = tid; i < rn * cq; i += 256) {
            const int r = i / cq, c4 = i - r * cq;
            *reinterpret_cast<float4*>(xs + r * ld + c4 * 4) = __ldg(src + i);
        }
        __syncthreads();
        // thread = (row, half of the channel quads); the two halves are adjacent lanes
        const int r = tid >> 1, h = tid & 1;
        float acc[16];
#pragma unroll
        for (int o = 0; o < 16; ++o) acc[o] = 0.f;
        if (r < rn) {
            for (int c4 = h; c4 < cq; c4 += 2) {
                const float4 v = *reinterpret_cast<const float4*>(xs + r * ld + c4 * 4);
#pragma unroll
                for (int o = 0; o < 16; ++o) {
                    if (o < cout) {
                        const float4 q = *reinterpret_cast<const float4*>(ws + o * cin + c4 * 4);
                        acc[o] = fmaf(v.x, q.x, fmaf(v.y, q.y, fmaf(v.z, q.z, fmaf(v.w, q.w, acc[o]))));
                    }
                }
            }
        }
#pragma unroll
        for (int o = 0; o < 16; ++o) acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 1);
        if (r < rn && h == 0) {
#pragma unroll
            for (int o = 0; o < 16; ++o) if (o < cout) os[r * cout + o] = acc[o] + (bias ? __ldg(bias + o) : 0.f);
        }
        __syncthreads();
        float* dst = y + r0 * cout;
        for (int i = tid; i < rn * cout; i += 256) dst[i] = accumulate ? dst[i] + os[i] : os[i];
    }
}

// block = 256 threads = `lanes` row lanes x cpad output channels (cpad = cout rounded up to 32); each thread keeps dw[co][0..cin)
// for its co in registers.  part: [gridDim.x][cout][cin], bpart: [gridDim.x][cout] (may be null).
__global__ void __launch_bounds__(256) wgrad_skinny_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                           float* __restrict__ part, float* __restrict__ bpart,
                                                           long long rows, int cin, int cout, int cpad) {
    extern __shared__ __align__(16) float sm[];
    float* xs = sm;                                  // [128][cin]
    float* red = xs + kSkinnyRows * 16;              // [lanes][cpad][17]
    const int tid = threadIdx.x;
    const int lanes = 256 / cpad;
    const int co = tid % cpad, rl = tid / cpad;
    const bool on = (co < cout) && (rl < lanes);
    float acc[16], bsum = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    const long long per = ((rows + gridDim.x - 1) / gridDim.x + kSkinnyRows - 1) / kSkinnyRows * kSkinnyRows;
    const long long rb = (long long)blockIdx.x * per;
    long long re = rb + per; if (re > rows) re = rows;
    for (long long r0 = rb; r0 < re; r0 += kSkinnyRows) {
        const int rn = (re - r0) < kSkinnyRows ? (int)(re - r0) : kSkinnyRows;
        __syncthreads();
        for (int i = tid; i < rn * cin; i += 256) xs[i] = __ldg(x + r0 * cin + i);
        __syncthreads();
        if (on) {
            for (int r = rl; r < rn; r += lanes) {
                const float d = __ldg(dy + (r0 + r) * cout + co);
                bsum += d;
#pragma unroll
                for (int i = 0; i < 16; ++i) if (i < cin) acc[i] = fmaf(d, xs[r * cin + i], acc[i]);
            }
        }
    }
    __syncthreads();
    if (rl < lanes) {
#pragma unroll
        for (int i = 0; i < 16; ++i) red[(rl * cpad + co) * 17 + i] = acc[i];
        red[(rl * cpad + co) * 17 + 16] = bsum;
    }
    __syncthreads();
    for (int o = tid; o < cout * 17; o += 256) {
        const int c = o / 17, i = o - c * 17;
        float s = 0.f;
        for (int l = 0; l < lanes; ++l) s += red[(l * cpad + c) * 17 + i];
        if (i < cin) part[((long long)blockIdx.x * cout + c) * cin + i] = s;
        else if (i == 16 && bpart != nullptr) bpart[(long long)blockIdx.x * cout + c] = s;
    }
}

// Vectorised variant for cout % 4 == 0: a thread owns FOUR consecutive output channels of one row lane, so every dy access is a
// 16-byte load, and four rows are fetched before the dependent FMAs (the scalar one-load-per-iteration loop above left the
// first unit's weight gradients at ~0.8 TB/s, profiles/r2a).  CMAX = register bound on cin (4 or 16).
// part: [gridDim.x][cout][cin], bpart: [gridDim.x][cout] (may be null).  Shared: xs[128][cin] | red[lanes][cout][CMAX + 1].
template <int CMAX>
__global__ void __launch_bounds__(256) wgrad_skinny4_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                            float* __restrict__ part, float* __restrict__ bpart,
                                                            long long rows, int cin, int cout) {
    extern __shared__ __align__(16) float sm[];
    float* xs = sm;                                  // [128][cin]
    float* red = xs + kSkinnyRows * 16;              // [lanes][cout][CMAX + 1]
    const int tid = threadIdx.x;
    const int cq = cout >> 2;
    const int lanes = 256 / cq;
    const int q = tid % cq, rl = tid / cq;
    const bool on = rl < lanes;
    float acc[4][CMAX], bsum[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        bsum[c] = 0.f;
#pragma unroll
        for (int i = 0; i < CMAX; ++i) acc[c][i] = 0.f;
    }
    const long long per = ((rows + gridDim.x - 1) / gridDim.x + kSkinnyRows - 1) / kSkinnyRows * kSkinnyRows;
    const long long rb = (long long)blockIdx.x * per;
    long long re = rb + per; if (re > rows) re = rows;
    for (long long r0 = rb; r0 < re; r0 += kSkinnyRows) {
        const int rn = (re - r0) < kSkinnyRows ? (int)(re - r0) : kSkinnyRows;
        __syncthreads();
        for (int i = tid; i < rn * cin; i += 256) xs[i] = __ldg(x + r0 * cin + i);
        __syncthreads();
        if (on) {
            const float4* src = reinterpret_cast<const float4*>(dy + r0 * cout) + q;
            for (int r = rl; r < rn; r += 4 * lanes) {
                float4 d[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rr = r + j * lanes;
                    d[j] = rr < rn ? __ldg(src + (long long)rr * cq) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rr = r + j * lanes;
                    if (rr < rn) {
                        bsum[0] += d[j].x; bsum[1] += d[j].y; bsum[2] += d[j].z; bsum[3] += d[j].w;
#pragma unroll
                        for (int i = 0; i < CMAX; ++i)
                            if (i < cin) {
                                const float xv = xs[rr * cin + i];
                                acc[0][i] = fmaf(d[j].x, xv, acc[0][i]); acc[1][i] = fmaf(d[j].y, xv, acc[1][i]);
                                acc[2][i] = fmaf(d[j].z, xv, acc[2][i]); acc[3][i] = fmaf(d[j].w, xv, acc[3][i]);
                            }
                    }
                }
            }
        }
    }
    __syncthreads();
    constexpr int LD = CMAX + 1;
    if (on) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float* dst = red + ((long long)rl * cout + q * 4 + c) * LD;
#pragma unroll
            for (int i = 0; i < CMAX; ++i) dst[i] = acc[c][i];
            dst[CMAX] = bsum[c];
        }
    }
    __syncthreads();
    for (int o = tid; o < cout * LD; o += 256) {
        const int c = o / LD, i = o - c * LD;
        float s = 0.f;
        for (int l = 0; l < lanes; ++l) s += red[((long long)l * cout + c) * LD + i];
        if (i < cin) part[((long long)blockIdx.x * cout + c) * cin + i] = s;
        else if (i == CMAX && bpart != nullptr) bpart[(long long)blockIdx.x * cout + c] = s;
    }
}

// column sums of dy for the bias gradient when the weight gradient runs on tensor cores: part[P][cout]
__global__ void __launch_bounds__(256) bias_partial_kernel(const float* dy, long long rows, int cout, float* part) {
    __shared__ float sm[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.y * 32 + tx;
    const long long per = (rows + gridDim.x - 1) / gridDim.x;
    const long long r0 = (long long)blockIdx.x * per;
    long long r1 = r0 + per; if (r1 > rows) r1 = rows;
    float s = 0.f;
    if (c < cout)
        for (long long r = r0 + ty; r < r1; r += 8) s += __ldg(dy + r * cout + c);
    sm[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && c < cout) {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc += sm[i][tx];
        part[(long long)blockIdx.x * cout + c] = acc;
    }
}

// the same column sums with 16-byte loads: thread = (row lane, channel quad), four rows in flight (cout % 4 == 0, cout / 4 <= 256)
__global__ void __launch_bounds__(256) bias_partial_vec_kernel(const float* __restrict__ dy, long long rows, int cout, float* __restrict__ part) {
    extern __shared__ __align__(16) float bsm[];      // [lanes_r][cout]
    const int cq = cout >> 2;
    const int lanes_r = 256 / cq;
    const int q = threadIdx.x % cq, rl = threadIdx.x / cq;
    const long long per = (rows + gridDim.x - 1) / gridDim.x;
    const long long r0 = (long long)blockIdx.x * per;
    long long r1 = r0 + per; if (r1 > rows) r1 = rows;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rl < lanes_r) {
        const float4* src = reinterpret_cast<const float4*>(dy) + q;
        for (long long r = r0 + rl; r < r1; r += 4LL * lanes_r) {
            float4 v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const long long rr = r + (long long)j * lanes_r;
                v[j] = rr < r1 ? __ldg(src + rr * cq) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) { s.x += v[j].x; s.y += v[j].y; s.z += v[j].z; s.w += v[j].w; }
        }
        *reinterpret_cast<float4*>(bsm + (size_t)rl * cout + q * 4) = s;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < cout; c += 256) {
        float acc = 0.f;
        for (int l = 0; l < lanes_r; ++l) acc += bsm[(size_t)l * cout + c];
        part[(long long)blockIdx.x * cout + c] = acc;
    }
}

constexpr int kBiasPartials = 2 * kNumSMs;

static int wgrad_splits(long long rows, int cin, int cout, int taps) {
    long long tiles = (long long)((cout + 63) / 64) * ((cin + 63) / 64) * taps;
    long long s = (4LL * kNumSMs + tiles - 1) / tiles;
    long long max_s = rows / 256;
    if (s > max_s) s = max_s;
    if (s > 64) s = 64;
    if (s < 1) s = 1;
    return (int)s;
}

}  // namespace agcn

using namespace agcn;

// implemented in conv_tc2.cu / wgrad_tc.cu; return AGCN_ERR_UNSUPPORTED when the shape is outside the tensor-core path
int agcn_conv_fwd_tc2(const float* x, const float* w, const float* bias, float* y,
                      int nb, int t_in, int t_out, int v, int cin, int cout,
                      int taps, int stride, int pad, int transposed, int accumulate, int split, float* w_split, void* stream,
                      float* stat_part, int* stat_nparts, const agcn::PostOp* post);
size_t agcn_conv_wgrad_tc_workspace_floats(int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad, int split);
int agcn_conv_wgrad_tc(const float* dy, const float* x, float* ws, int* splits_out,
                       int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad, int split, void* stream);
int agcn_conv_wgrad_tc_presplit(const uint16_t* dy_split, const uint16_t* x_split, float* ws, int* splits_out,
                                int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad, void* stream);

static bool known_precision(int p) { return p >= AGCN_PREC_FP32 && p <= AGCN_PREC_BF16X3; }

extern "C" AGCN_API size_t agcn_conv_fwd_workspace_bytes(int cin, int cout, int taps, int precision) {
    if ((precision != AGCN_PREC_FP32 && precision != AGCN_PREC_BF16X3) || cin <= 0 || cout <= 0 || taps <= 0) return 0;
    // strict mode: rna_tf32(w) as fp32 followed by the bf16 [hi16 | lo16] cross rows of every 32-channel K chunk (padded to whole
    // chunks); the BF16x3 path needs less (bf16 h | m) and falls back to the strict kernels for channel counts not a multiple of 16
    const size_t nchunk = (size_t)(cin + 31) / 32;
    return (size_t)cout * taps * cin * sizeof(float) + (size_t)cout * taps * nchunk * 128;
}

static int conv_fwd_impl(const float* x, const float* w, const float* bias, float* y,
                         int nb, int t_in, int t_out, int v, int cin, int cout,
                         int taps, int stride, int pad, int transposed, int accumulate,
                         int precision, void* workspace, size_t workspace_bytes, void* stream,
                         float* stat_part, int* stat_nparts, const PostOp* post = nullptr) {
    AGCN_REQUIRE(x && w && y, AGCN_ERR_NULL, "agcn_conv_fwd: null pointer");
    AGCN_REQUIRE(nb > 0 && t_in > 0 && t_out > 0 && v > 0 && cin > 0 && cout > 0 && taps > 0 && stride > 0 && pad >= 0,
                 AGCN_ERR_BAD_SHAPE, "agcn_conv_fwd: bad shape nb=%d t_in=%d t_out=%d v=%d cin=%d cout=%d taps=%d stride=%d pad=%d",
                 nb, t_in, t_out, v, cin, cout, taps, stride, pad);
    AGCN_REQUIRE(known_precision(precision), AGCN_ERR_UNSUPPORTED, "agcn_conv_fwd: unknown precision %d", precision);
    if (precision == AGCN_PREC_TF32 || precision == AGCN_PREC_FP32 || precision == AGCN_PREC_BF16X3) {
        const int first_split = precision == AGCN_PREC_FP32 ? 1 : (precision == AGCN_PREC_BF16X3 ? 2 : 0);
        for (int split = first_split; split >= (first_split == 2 ? 1 : first_split); --split) {      // BF16x3 falls back to 3xTF32
        const bool ws_ok = !split || (workspace != nullptr && workspace_bytes >= agcn_conv_fwd_workspace_bytes(cin, cout, taps, precision));
        if (ws_ok) {
            if (stat_part != nullptr) {       // try the epilogue with fused column sums first; shapes it does not take run without
                int rc3 = agcn_conv_fwd_tc2(x, w, bias, y, nb, t_in, t_out, v, cin, cout, taps, stride, pad, transposed, accumulate, split,
                                            static_cast<float*>(workspace), stream, stat_part, stat_nparts, post);
                if (rc3 != AGCN_ERR_UNSUPPORTED) return rc3;
            }
            int rc2 = agcn_conv_fwd_tc2(x, w, bias, y, nb, t_in, t_out, v, cin, cout, taps, stride, pad, transposed, accumulate, split,
                                        static_cast<float*>(workspace), stream, nullptr, nullptr, post);
            if (rc2 != AGCN_ERR_UNSUPPORTED) return rc2;   // unsupported shapes fall through to the FFMA kernel
        }
        }
    }
    if (post == nullptr && taps == 1 && stride == 1 && pad == 0 && t_in == t_out && cout < 16 && cin % 4 == 0 && cin <= 1024 && aligned16(x) && aligned16(w)) {
        // skinny output (input gradients of the first unit): one HBM pass, no GEMM tiling
        const long long rows = (long long)nb * t_out * v;
        const size_t smem = ((size_t)kSkinnyRows * (cin + 4) + (size_t)cout * cin + (size_t)kSkinnyRows * cout) * sizeof(float);
        if (smem <= 200 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(conv_skinny_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            if (e != cudaSuccess) return fail(AGCN_ERR_CUDA, "agcn_conv_fwd: %s", cudaGetErrorString(e));
            long long blocks = (rows + kSkinnyRows - 1) / kSkinnyRows;
            if (blocks > 8LL * kNumSMs) blocks = 8LL * kNumSMs;
            conv_skinny_out_kernel<<<(unsigned)blocks, 256, smem, static_cast<cudaStream_t>(stream)>>>(x, w, bias, y, rows, cin, cout, accumulate);
            return check_launch("agcn_conv_fwd(skinny)");
        }
    }
    ConvArgs a{x, w, bias, y, nb, t_in, t_out, v, cin, cout, taps, stride, pad, transposed, accumulate,
               (long long)nb * t_out * v, post ? *post : PostOp{nullptr, nullptr, nullptr, 0}};
    dim3 grid((unsigned)ceil_div(a.rows_out, 128), (unsigned)ceil_div(cout, 64));
    const bool vec = (cin % 4 == 0) && aligned16(x) && aligned16(w);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (vec) conv_fwd_kernel<true><<<grid, 256, 0, s>>>(a);
    else conv_fwd_kernel<false><<<grid, 256, 0, s>>>(a);
    return check_launch("agcn_conv_fwd");
}

extern "C" AGCN_API int agcn_conv_fwd(const float* x, const float* w, const float* bias, float* y,
                             int nb, int t_in, int t_out, int v, int cin, int cout,
                             int taps, int stride, int pad, int transposed, int accumulate,
                             int precision, void* workspace, size_t workspace_bytes, void* stream) {
    return conv_fwd_impl(x, w, bias, y, nb, t_in, t_out, v, cin, cout, taps, stride, pad, transposed, accumulate, precision,
                         workspace, workspace_bytes, stream, nullptr, nullptr);
}

extern "C" AGCN_API int agcn_conv_fwd_post(const float* x, const float* w, const float* bias,
                                           const float* scale, const float* shift, const float* res, int relu, float* y,
                                           int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad,
                                           int precision, void* workspace, size_t workspace_bytes, void* stream) {
    AGCN_REQUIRE((scale == nullptr) == (shift == nullptr), AGCN_ERR_NULL, "agcn_conv_fwd_post: scale and shift come together");
    AGCN_REQUIRE(!scale || (aligned16(scale) && aligned16(shift)), AGCN_ERR_MISALIGNED, "agcn_conv_fwd_post: scale / shift not 16-byte aligned");
    AGCN_REQUIRE(!res || aligned16(res), AGCN_ERR_MISALIGNED, "agcn_conv_fwd_post: residual tensor not 16-byte aligned");
    PostOp post{scale, shift, res, relu};
    return conv_fwd_impl(x, w, bias, y, nb, t_in, t_out, v, cin, cout, taps, stride, pad, 0, 0, precision,
                         workspace, workspace_bytes, stream, nullptr, nullptr, &post);
}

extern "C" AGCN_API size_t agcn_conv_fwd_stats_bytes(int cout) {
    return cout > 0 ? (size_t)4 * kNumSMs * 4 * cout * sizeof(float) : 0;       // [4 warps x SMs][shifted sum | sum of squares | pivot | rows][cout]
}

extern "C" AGCN_API int agcn_conv_fwd_stats(const float* x, const float* w, const float* bias, float* y,
                                   int nb, int t_in, int t_out, int v, int cin, int cout,
                                   int taps, int stride, int pad,
                                   int precision, void* workspace, size_t workspace_bytes,
                                   float* stat_part, size_t stat_part_bytes, int* stat_nparts, void* stream) {
    AGCN_REQUIRE(stat_part && stat_nparts, AGCN_ERR_NULL, "agcn_conv_fwd_stats: null pointer");
    AGCN_REQUIRE(cout > 0 && stat_part_bytes >= agcn_conv_fwd_stats_bytes(cout), AGCN_ERR_WORKSPACE, "agcn_conv_fwd_stats: partial buffer too small");
    AGCN_REQUIRE(aligned16(stat_part), AGCN_ERR_MISALIGNED, "agcn_conv_fwd_stats: partial buffer not 16-byte aligned");
    *stat_nparts = 0;
    static const bool off = probe_env("AGCN_NO_FUSED_STATS") != nullptr;
    return conv_fwd_impl(x, w, bias, y, nb, t_in, t_out, v, cin, cout, taps, stride, pad, 0, 0, precision,
                         workspace, workspace_bytes, stream, off ? nullptr : stat_part, off ? nullptr : stat_nparts);
}

extern "C" AGCN_API size_t agcn_conv_wgrad_workspace_bytes(int nb, int t_in, int t_out, int v, int cin, int cout, int taps) {
    long long rows = (long long)nb * t_out * v;
    int splits = wgrad_splits(rows, cin, cout, taps);
    size_t simt = (size_t)splits * ((size_t)cout * taps * cin + (size_t)cout);
    const int pad = (taps - 1) / 2;
    size_t tc = 0;
    for (int stride = 1; stride <= 2; ++stride)
        for (int split = 0; split <= 2; ++split) {
            size_t f = agcn_conv_wgrad_tc_workspace_floats(nb, t_in, t_out, v, cin, cout, taps, stride, pad, split);
            if (f > tc) tc = f;
        }
    tc += (size_t)kBiasPartials * cout;
    const size_t skinny = (taps == 1 && cin <= 16) ? (size_t)4 * kNumSMs * ((size_t)cout * cin + cout) : 0;
    size_t need = simt > tc ? simt : tc;
    if (skinny > need) need = skinny;
    return need * sizeof(float);
}

// Weight gradient from operands that arrive split into bf16 pieces: dy_split [2][nb*t_out*v][cout] and x_split [2][nb*t_in*v][cin]
// (plane 0 = h = bf16(value), plane 1 = m = bf16(value - h), round to nearest), as written by agcn_bn_apply /
// agcn_bn_bwd (out_split / dy_split).  Same arithmetic as the parity modes of agcn_conv_wgrad (h.h + h.m + m.h on kind::f16) without the
// in-kernel conversion.  No bias gradient.  AGCN_ERR_UNSUPPORTED (quiet) for channel counts that are not multiples of 64: use
// agcn_conv_wgrad on the fp32 tensors then.
extern "C" AGCN_API int agcn_conv_wgrad_presplit(const void* dy_split, const void* x_split, float* dw,
                                                 int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad,
                                                 void* workspace, size_t workspace_bytes, void* stream) {
    AGCN_REQUIRE(dy_split && x_split && dw && workspace, AGCN_ERR_NULL, "agcn_conv_wgrad_presplit: null pointer");
    AGCN_REQUIRE(nb > 0 && t_in > 0 && t_out > 0 && v > 0 && cin > 0 && cout > 0 && taps > 0 && stride > 0 && pad >= 0, AGCN_ERR_BAD_SHAPE,
                 "agcn_conv_wgrad_presplit: bad shape");
    AGCN_REQUIRE(workspace_bytes >= agcn_conv_wgrad_workspace_bytes(nb, t_in, t_out, v, cin, cout, taps), AGCN_ERR_WORKSPACE,
                 "agcn_conv_wgrad_presplit: workspace too small");
    AGCN_REQUIRE(aligned16(workspace), AGCN_ERR_MISALIGNED, "agcn_conv_wgrad_presplit: workspace not 16-byte aligned");
    float* ws = static_cast<float*>(workspace);
    int splits = 0;
    int rc = agcn_conv_wgrad_tc_presplit(static_cast<const uint16_t*>(dy_split), static_cast<const uint16_t*>(x_split), ws, &splits,
                                         nb, t_in, t_out, v, cin, cout, taps, stride, pad, stream);
    if (rc) return rc;
    const long long wsize = (long long)cout * taps * cin;
    wgrad_reduce_kernel<<<ceil_div(wsize, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(ws, nullptr, dw, nullptr, wsize, cout, splits);
    return check_launch("agcn_conv_wgrad_presplit(reduce)");
}

extern "C" AGCN_API int agcn_conv_wgrad(const float* dy, const float* x, float* dw, float* dbias,
                               int nb, int t_in, int t_out, int v, int cin, int cout,
                               int taps, int stride, int pad,
                               void* workspace, size_t workspace_bytes, int precision, void* stream) {
    AGCN_REQUIRE(dy && x && dw && workspace, AGCN_ERR_NULL, "agcn_conv_wgrad: null pointer");
    AGCN_REQUIRE(nb > 0 && t_in > 0 && t_out > 0 && v > 0 && cin > 0 && cout > 0 && taps > 0 && stride > 0 && pad >= 0,
                 AGCN_ERR_BAD_SHAPE, "agcn_conv_wgrad: bad shape");
    const size_t need = agcn_conv_wgrad_workspace_bytes(nb, t_in, t_out, v, cin, cout, taps);
    AGCN_REQUIRE(workspace_bytes >= need, AGCN_ERR_WORKSPACE, "agcn_conv_wgrad: workspace %zu < %zu", workspace_bytes, need);
    AGCN_REQUIRE(aligned16(workspace), AGCN_ERR_MISALIGNED, "agcn_conv_wgrad: workspace not 16-byte aligned");
    AGCN_REQUIRE(known_precision(precision), AGCN_ERR_UNSUPPORTED, "agcn_conv_wgrad: unknown precision %d", precision);
    // Both parity modes take the BF16x3 weight-gradient kernel: a weight gradient is a LEAF of the backward pass, so its ~1e-5
    // error (bf16 h + m pieces, three products) stays in that one tensor instead of compounding through the layers the way the
    // forward / input-gradient contractions' error does (measured: whole-model gradients 8e-6 with only the weight gradients on
    // BF16x3, 1.5e-4 with the temporal convolutions on it too).  20-25 % faster than the 3xTF32 kernel.
    int tc_split = (precision == AGCN_PREC_FP32 || precision == AGCN_PREC_BF16X3) ? 2 : 0;
    size_t tc_floats = precision == AGCN_PREC_FP32_FFMA ? 0 :
        agcn_conv_wgrad_tc_workspace_floats(nb, t_in, t_out, v, cin, cout, taps, stride, pad, tc_split);
    if (tc_floats == 0 && tc_split == 2) {          // shape outside the BF16x3 plan: the 3xTF32 kernel is the other parity path
        tc_split = 1;
        tc_floats = agcn_conv_wgrad_tc_workspace_floats(nb, t_in, t_out, v, cin, cout, taps, stride, pad, tc_split);
    }
    if (tc_floats > 0 && (tc_floats + (size_t)kBiasPartials * cout) * sizeof(float) <= workspace_bytes) {
        float* ws = static_cast<float*>(workspace);
        int tc_splits = 0;
        int rc = agcn_conv_wgrad_tc(dy, x, ws, &tc_splits, nb, t_in, t_out, v, cin, cout, taps, stride, pad, tc_split, stream);
        if (rc == AGCN_OK) {
            cudaStream_t s = static_cast<cudaStream_t>(stream);
            const long long wsize = (long long)cout * taps * cin;
            wgrad_reduce_kernel<<<ceil_div(wsize, 256), 256, 0, s>>>(ws, nullptr, dw, nullptr, wsize, cout, tc_splits);
            rc = check_launch("agcn_conv_wgrad(tc reduce)");
            if (rc) return rc;
            if (dbias) {
                float* part = ws + (size_t)tc_splits * wsize;
                const long long rows = (long long)nb * t_out * v;
                int P = (int)((rows + 255) / 256);
                if (P > kBiasPartials) P = kBiasPartials;
                if (cout % 4 == 0 && cout / 4 <= 256 && aligned16(dy)) {
                    const size_t bsmem = (size_t)(256 / (cout / 4)) * cout * sizeof(float);
                    bias_partial_vec_kernel<<<P, 256, bsmem, s>>>(dy, rows, cout, part);
                } else {
                    dim3 grid((unsigned)P, (unsigned)ceil_div(cout, 32));
                    bias_partial_kernel<<<grid, 256, 0, s>>>(dy, rows, cout, part);
                }
                rc = check_launch("agcn_conv_wgrad(bias partial)");
                if (rc) return rc;
                wgrad_reduce_kernel<<<ceil_div(cout, 256), 256, 0, s>>>(nullptr, part, nullptr, dbias, 0, cout, P);
                rc = check_launch("agcn_conv_wgrad(bias reduce)");
            }
            return rc;
        }
        if (rc != AGCN_ERR_UNSUPPORTED) return rc;      // unsupported shapes fall through to the FFMA kernel
    }
    if (taps == 1 && stride == 1 && pad == 0 && t_in == t_out && cin <= 16 && cout <= 256 &&
        (cin % 4 != 0 || cout % 4 != 0 || precision != AGCN_PREC_TF32)) {      // TF32 mode keeps tensor-core-eligible shapes on the tensor cores
        // skinny input (weight gradients of the first unit)
        const long long rows = (long long)nb * t_out * v;
        const int cpad = (cout + 31) / 32 * 32;
        const int lanes = 256 / cpad;
        long long P = (rows + 4 * kSkinnyRows - 1) / (4 * kSkinnyRows);
        if (P > 4LL * kNumSMs) P = 4LL * kNumSMs;
        if (P < 1) P = 1;
        const long long wsize = (long long)cout * cin;
        if ((size_t)P * (wsize + cout) * sizeof(float) <= workspace_bytes) {
            float* part = static_cast<float*>(workspace);
            float* bpart = dbias ? part + P * wsize : nullptr;
            const size_t smem = ((size_t)kSkinnyRows * 16 + (size_t)lanes * cpad * 17) * sizeof(float);
            cudaStream_t s = static_cast<cudaStream_t>(stream);
            static const bool scalar_only = probe_env("AGCN_SKINNY_SCALAR") != nullptr;
            const int cmax = cin <= 4 ? 4 : 16;
            const size_t smem4 = ((size_t)kSkinnyRows * 16 + (size_t)(256 / (cout / 4 > 0 ? cout / 4 : 1)) * cout * (cmax + 1)) * sizeof(float);
            if (!scalar_only && cout % 4 == 0 && cout >= 16 && aligned16(dy) && smem4 <= 100 * 1024) {
                cudaError_t e = cmax == 4 ? cudaFuncSetAttribute(wgrad_skinny4_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)
                                          : cudaFuncSetAttribute(wgrad_skinny4_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
                if (e != cudaSuccess) return fail(AGCN_ERR_CUDA, "agcn_conv_wgrad: %s", cudaGetErrorString(e));
                if (cmax == 4) wgrad_skinny4_kernel<4><<<(unsigned)P, 256, smem4, s>>>(dy, x, part, bpart, rows, cin, cout);
                else wgrad_skinny4_kernel<16><<<(unsigned)P, 256, smem4, s>>>(dy, x, part, bpart, rows, cin, cout);
            } else {
                wgrad_skinny_kernel<<<(unsigned)P, 256, smem, s>>>(dy, x, part, bpart, rows, cin, cout, cpad);
            }
            int rc = check_launch("agcn_conv_wgrad(skinny)");
            if (rc) return rc;
            const long long total = wsize + (dbias ? cout : 0);
            wgrad_reduce_kernel<<<ceil_div(total, 256), 256, 0, s>>>(part, bpart, dw, dbias, wsize, cout, (int)P);
            return check_launch("agcn_conv_wgrad(skinny reduce)");
        }
    }
    WgradArgs a;
    a.dy = dy; a.x = x;
    a.nb = nb; a.t_in = t_in; a.t_out = t_out; a.v = v; a.cin = cin; a.cout = cout;
    a.taps = taps; a.stride = stride; a.pad = pad;
    a.rows_out = (long long)nb * t_out * v;
    const int splits = wgrad_splits(a.rows_out, cin, cout, taps);
    long long rps = (a.rows_out + splits - 1) / splits;
    rps = (rps + 31) / 32 * 32;
    a.rows_per_split = rps;
    a.ntiles = (cout + 63) / 64; a.ktiles = (cin + 63) / 64;
    const long long wsize = (long long)cout * taps * cin;
    a.ws_w = static_cast<float*>(workspace);
    a.ws_b = dbias ? a.ws_w + (long long)splits * wsize : nullptr;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    dim3 grid((unsigned)(a.ntiles * a.ktiles * taps), (unsigned)splits);
    const bool vec = (cin % 4 == 0) && (cout % 4 == 0) && aligned16(x) && aligned16(dy);
    if (vec) conv_wgrad_kernel<true><<<grid, 256, 0, s>>>(a);
    else conv_wgrad_kernel<false><<<grid, 256, 0, s>>>(a);
    int rc = check_launch("agcn_conv_wgrad");
    if (rc) return rc;
    const long long total = wsize + (dbias ? cout : 0);
    wgrad_reduce_kernel<<<ceil_div(total, 256), 256, 0, s>>>(a.ws_w, a.ws_b, dw, dbias, wsize, cout, splits);
    return check_launch("agcn_conv_wgrad(reduce)");
}
