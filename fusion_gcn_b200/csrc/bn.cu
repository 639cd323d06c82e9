// BatchNorm statistics / apply / backward, and the global mean pool, on channels-last tensors.
// Reference arithmetic: nn.BatchNorm2d / nn.BatchNorm1d in training mode (torch_src/models/mmargcn/agcn.py:44,78,83,150),
// ReLU + residual adds (:113-115, :135-136), mean pooling (:194-196).
// Reductions are two-phase and deterministic: per-CTA fp32 partials in a fixed row partition, combined in fp64.
#include "common.cuh"
#include <initializer_list>

namespace agcn {

constexpr int kMaxPartials = 4 * kNumSMs;   // 592

struct RowMap {
    int outer, inner; long long outer_stride; int channels;
    __device__ __forceinline__ long long row_offset(long long r) const {
        if (outer == 1) return r * channels;
        long long o = r / inner;
        return o * outer_stride + (r - o * inner) * channels;
    }
};

static int num_partials(long long rows) {
    long long p = (rows + 63) / 64;
    if (p > kMaxPartials) p = kMaxPartials;
    if (p < 1) p = 1;
    return (int)p;
}

// NS sums per channel.  MODE 0: (x - pivot, (x - pivot)^2) with the per-channel pivot passed in `mean` (NULL: 0) -- shifted sums, so
// that var = E[(x-p)^2] - E[x-p]^2 does not cancel for channels with |mean| >> sigma.  MODE 1: (g, g*xhat) with g = dout * [mask > 0].
// grid = (P, column strips of 32); block = 32 columns x 8 row lanes.
template <int MODE>
__global__ void __launch_bounds__(256) colsum_strip_kernel(const float* x, const float* dout, const float* mask,
                                                           const float* mean, const float* invstd,
                                                           RowMap m, long long rows, float* part) {
    __shared__ float sm[2][8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.y * 32 + tx;
    const int P = gridDim.x;
    const long long per = (rows + P - 1) / P;
    const long long r0 = (long long)blockIdx.x * per;
    long long r1 = r0 + per; if (r1 > rows) r1 = rows;
    float s0 = 0.f, s1 = 0.f;
    if (c < m.channels) {
        float mu = 0.f, is = 0.f;
        if (MODE == 1) { mu = mean[c]; is = invstd[c]; }
        else if (mean != nullptr) mu = mean[c];
        for (long long r = r0 + ty; r < r1; r += 8) {
            const long long off = m.row_offset(r) + c;
            if (MODE == 0) {
                float v = __ldg(x + off) - mu;
                s0 += v; s1 = fmaf(v, v, s1);
            } else {
                float g = __ldg(dout + off);
                if (mask != nullptr && !(__ldg(mask + off) > 0.f)) g = 0.f;
                float xh = (__ldg(x + off) - mu) * is;
                s0 += g; s1 = fmaf(g, xh, s1);
            }
        }
    }
    sm[0][ty][tx] = s0; sm[1][ty][tx] = s1;
    __syncthreads();
    if (ty == 0 && c < m.channels) {
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) { a += sm[0][i][tx]; b += sm[1][i][tx]; }
        part[((long long)blockIdx.x * 2 + 0) * m.channels + c] = a;
        part[((long long)blockIdx.x * 2 + 1) * m.channels + c] = b;
    }
}

// Vectorised variant for channels % 4 == 0 and 256 % (channels/4) == 0 (64, 128, 256, ...; outer == 1 or not).
// mask_bits (MODE 1, contiguous rows only): the ReLU mask as one bit per element, bit (e & 31) of word e >> 5 for the linear element
// index e = row * channels + c, written by bn_apply_kernel -- read instead of the fp32 mask tensor (1/32 of the bytes).
__device__ __forceinline__ unsigned mask_nibble(const unsigned* bits, long long off) {
    return (__ldg(bits + (off >> 5)) >> (unsigned)(off & 31)) & 0xFu;
}

// bcast_rows > 0 (MODE 1): dout is the gradient of a fused mean pool, [groups][channels]; element (r, c) reads
// dout[r / bcast_rows][c] * bcast_scale (agcn_bn_bwd with pool_rows > 0).
template <int MODE>
__global__ void __launch_bounds__(256) colsum_vec_kernel(const float* x, const float* dout, const float* mask, const unsigned* mask_bits,
                                                         const float* mean, const float* invstd,
                                                         RowMap m, long long rows, float* part, int bcast_rows = 0, float bcast_scale = 1.f) {
    extern __shared__ __align__(16) float smv[];   // [2][lanes_r][channels]
    const int cq = m.channels >> 2;
    const int lanes_r = 256 / cq;
    const int q = threadIdx.x % cq, rl = threadIdx.x / cq;
    const int P = gridDim.x;
    const long long per = (rows + P - 1) / P;
    const long long r0 = (long long)blockIdx.x * per;
    long long r1 = r0 + per; if (r1 > rows) r1 = rows;
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
    float4 mu = s0, is = s0;
    if (MODE == 1) {
        mu = *reinterpret_cast<const float4*>(mean + q * 4);
        is = *reinterpret_cast<const float4*>(invstd + q * 4);
    } else if (mean != nullptr) {
        mu = *reinterpret_cast<const float4*>(mean + q * 4);       // MODE 0: the pivot of the shifted sums
    }
    // U rows per trip with every load issued before the first dependent add: 592 CTAs x 256 threads with one 16-byte load each in
    // flight cover only ~2.4 MB, a third of what the HBM latency-bandwidth product needs (the plain loop measured 3.2 TB/s, r8_stage);
    // the additions keep their row order, so the sums are bit-identical to the rolled loop's
    constexpr int U = MODE == 0 ? 4 : 2;
    auto body = [&](const float4& v_in, float4 g, unsigned nib, const float4& k, bool has_k) {
        if (MODE == 0) {
            float4 v = v_in;
            v.x -= mu.x; v.y -= mu.y; v.z -= mu.z; v.w -= mu.w;
            s0.x += v.x; s0.y += v.y; s0.z += v.z; s0.w += v.w;
            s1.x = fmaf(v.x, v.x, s1.x); s1.y = fmaf(v.y, v.y, s1.y); s1.z = fmaf(v.z, v.z, s1.z); s1.w = fmaf(v.w, v.w, s1.w);
        } else {
            if (bcast_rows > 0) { g.x *= bcast_scale; g.y *= bcast_scale; g.z *= bcast_scale; g.w *= bcast_scale; }
            if (mask_bits != nullptr) {
                if (!(nib & 1u)) g.x = 0.f;
                if (!(nib & 2u)) g.y = 0.f;
                if (!(nib & 4u)) g.z = 0.f;
                if (!(nib & 8u)) g.w = 0.f;
            } else if (has_k) {
                if (!(k.x > 0.f)) g.x = 0.f;
                if (!(k.y > 0.f)) g.y = 0.f;
                if (!(k.z > 0.f)) g.z = 0.f;
                if (!(k.w > 0.f)) g.w = 0.f;
            }
            const float4& v = v_in;
            s0.x += g.x; s0.y += g.y; s0.z += g.z; s0.w += g.w;
            s1.x = fmaf(g.x, (v.x - mu.x) * is.x, s1.x); s1.y = fmaf(g.y, (v.y - mu.y) * is.y, s1.y);
            s1.z = fmaf(g.z, (v.z - mu.z) * is.z, s1.z); s1.w = fmaf(g.w, (v.w - mu.w) * is.w, s1.w);
        }
    };
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    long long r = r0 + rl;
    for (; r + (long long)(U - 1) * lanes_r < r1; r += (long long)U * lanes_r) {
        float4 v[U], g[U], k[U];
        unsigned nib[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long ru = r + (long long)u * lanes_r;
            const long long off = m.row_offset(ru) + q * 4;
            v[u] = __ldg(reinterpret_cast<const float4*>(x + off));
            g[u] = zero4; k[u] = zero4; nib[u] = 0u;
            if (MODE == 1) {
                g[u] = bcast_rows > 0 ? __ldg(reinterpret_cast<const float4*>(dout + (ru / bcast_rows) * m.channels + q * 4))
                                      : __ldg(reinterpret_cast<const float4*>(dout + off));
                if (mask_bits != nullptr) nib[u] = mask_nibble(mask_bits, off);
                else if (mask != nullptr) k[u] = __ldg(reinterpret_cast<const float4*>(mask + off));
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) body(v[u], g[u], nib[u], k[u], mask != nullptr);
    }
    for (; r < r1; r += lanes_r) {
        const long long off = m.row_offset(r) + q * 4;
        const float4 v = __ldg(reinterpret_cast<const float4*>(x + off));
        float4 g = zero4, k = zero4;
        unsigned nib = 0u;
        if (MODE == 1) {
            g = bcast_rows > 0 ? __ldg(reinterpret_cast<const float4*>(dout + (r / bcast_rows) * m.channels + q * 4))
                               : __ldg(reinterpret_cast<const float4*>(dout + off));
            if (mask_bits != nullptr) nib = mask_nibble(mask_bits, off);
            else if (mask != nullptr) k = __ldg(reinterpret_cast<const float4*>(mask + off));
        }
        body(v, g, nib, k, mask != nullptr);
    }
    float4* a = reinterpret_cast<float4*>(smv);
    a[(0 * lanes_r + rl) * cq + q] = s0;
    a[(1 * lanes_r + rl) * cq + q] = s1;
    __syncthreads();
    // 2 * channels outputs, each summed over lanes_r
    for (int o = threadIdx.x; o < 2 * m.channels; o += 256) {
        const int which = o / m.channels, c = o % m.channels;
        float acc = 0.f;
        for (int i = 0; i < lanes_r; ++i) acc += smv[(which * lanes_r + i) * m.channels + c];
        part[((long long)blockIdx.x * 2 + which) * m.channels + c] = acc;
    }
}

// Sum of the P per-CTA partials of channel c (fp64, fixed order): kFinLanes lanes per channel stride over the partials, then a
// fixed-order shared-memory combine.  block = kFinCh channels x kFinLanes lanes: the finalize kernels are pure latency (a few
// hundred partials per channel, ~25 launches per step), so the partials are spread over many lanes and blocks.
constexpr int kFinCh = 8, kFinLanes = 32, kFinBatch = 10, kFinBatch4 = 10;
__device__ __forceinline__ void reduce_partials(const float* part, int P, int C, int c, double& s_out, double& q_out) {
    __shared__ double red[2][kFinLanes][kFinCh + 1];
    const int tx = threadIdx.x % kFinCh, ty = threadIdx.x / kFinCh;
    double s = 0.0, q = 0.0;
    if (c < C)
        // kFinBatch partials per trip, every load issued before the first add: the kernel is a chain of dependent round trips to
        // L2 / HBM (ncu r9: 11.7 us for 592 partials with four loads in flight) and sits between every column-sum pass and its apply pass
        for (int b0 = ty; b0 < P; b0 += kFinLanes * kFinBatch) {
            float vs[kFinBatch], vq[kFinBatch];
#pragma unroll
            for (int i = 0; i < kFinBatch; ++i) {
                const int b = b0 + i * kFinLanes;
                vs[i] = b < P ? part[((long long)b * 2 + 0) * C + c] : 0.f;
                vq[i] = b < P ? part[((long long)b * 2 + 1) * C + c] : 0.f;
            }
#pragma unroll
            for (int i = 0; i < kFinBatch; ++i) { s += (double)vs[i]; q += (double)vq[i]; }
        }
    red[0][ty][tx] = s; red[1][ty][tx] = q;
    __syncthreads();
    s = 0.0; q = 0.0;
#pragma unroll
    for (int i = 0; i < kFinLanes; ++i) { s += red[0][i][tx]; q += red[1][i][tx]; }
    s_out = s; q_out = q;
}

// The same for the partials of the convolution epilogue (agcn_conv_fwd_stats): part[P][4][C] = shifted sum | shifted sum of squares |
// pivot | row count per partial.  In fp64:  a = sum_p (n_p piv_p + s1_p) = sum x,   b = sum_p (s2_p + piv_p (2 s1_p + n_p piv_p)) = sum x^2
// (the same numbers as the pairwise-variance merge -- its s1^2 / n terms cancel -- without a division per partial); the caller forms
// var = b / N - (a / N)^2, whose cancellation costs (mean / sigma)^2 x 1e-16 in fp64, while the rounding of the fp32 partials enters
// through (piv_p - mean) ~ sigma, not through mean.
__device__ __forceinline__ void reduce_partials4(const float* part, int P, int C, int c, double& a_out, double& b_out) {
    __shared__ double red4[2][kFinLanes][kFinCh + 1];
    const int tx = threadIdx.x % kFinCh, ty = threadIdx.x / kFinCh;
    double a = 0.0, b = 0.0;
    if (c < C)
        // all loads of kFinBatch4 partials first (one round trip per batch); a warp that never saw this column left n = 0 and its pivot unwritten
        for (int p0 = ty; p0 < P; p0 += kFinLanes * kFinBatch4) {
            float f0[kFinBatch4], f1[kFinBatch4], f2[kFinBatch4], nf[kFinBatch4];
#pragma unroll
            for (int i = 0; i < kFinBatch4; ++i) {
                const int p = p0 + i * kFinLanes;
                const float* q = part + (long long)(p < P ? p : 0) * 4 * C + c;
                f0[i] = q[0]; f1[i] = q[C]; f2[i] = q[2 * C]; nf[i] = p < P ? q[3 * C] : -1.f;
            }
#pragma unroll
            for (int i = 0; i < kFinBatch4; ++i) {
                if (nf[i] < 0.f) continue;                   // past the last partial
                const double n = (double)nf[i], s1 = (double)f0[i], s2 = (double)f1[i], pv = nf[i] > 0.f ? (double)f2[i] : 0.0;
                a += n * pv + s1;
                b += s2 + pv * (2.0 * s1 + n * pv);
            }
        }
    red4[0][ty][tx] = a; red4[1][ty][tx] = b;
    __syncthreads();
    a = 0.0; b = 0.0;
#pragma unroll
    for (int i = 0; i < kFinLanes; ++i) { a += red4[0][i][tx]; b += red4[1][i][tx]; }
    a_out = a; b_out = b;
}

__global__ void __launch_bounds__(256) bn_finalize_kernel(const float* part, int P, int C, double count,
                                   const float* gamma, const float* beta, float* running_mean, float* running_var,
                                   long long* nbt, float momentum, float eps, int training,
                                   float* scale, float* shift, float* save_mean, float* save_invstd, const float* pivot, int layout4) {
    const int c = blockIdx.x * kFinCh + threadIdx.x % kFinCh;
    if (blockIdx.x == 0 && threadIdx.x == 0 && training && nbt != nullptr) *nbt += 1;
    double s = 0.0, q = 0.0;
    if (training) {
        if (layout4) reduce_partials4(part, P, C, c, s, q);
        else reduce_partials(part, P, C, c, s, q);
    }
    if (c >= C || threadIdx.x >= kFinCh) return;
    double mean, var;
    if (training) {
        if (layout4) {
            mean = s / count;
            var = q / count - mean * mean;
        } else {
            // the partials are sums of (x - pivot) and (x - pivot)^2 with one pivot for the whole tensor
            const double d = s / count;
            mean = (pivot != nullptr ? (double)pivot[c] : 0.0) + d;
            var = q / count - d * d;
        }
        if (var < 0.0) var = 0.0;
        if (running_mean != nullptr) {
            const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
            running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mean);
            running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
        }
    } else {
        mean = running_mean[c];
        var = running_var[c];
    }
    const double invstd = 1.0 / sqrt(var + (double)eps);
    const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    const float sc = (float)(g * invstd);
    scale[c] = sc;
    shift[c] = (float)(b - mean * g * invstd);
    if (save_mean) save_mean[c] = (float)mean;
    if (save_invstd) save_invstd[c] = (float)invstd;
}

// bf16 pieces of four fp32 values, as the parity modes' converters form them (tc_common.cuh bf16_split8): h = bf16(x), m = bf16(x - h),
// round to nearest (ties away), packed in channel order -- the operand format of agcn_conv_wgrad_presplit
__device__ __forceinline__ void bf16_pieces4(const float v[4], uint2& h, uint2& m) {
    unsigned hb[4], mb[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        hb[i] = (__float_as_uint(v[i]) + 0x8000u) & 0xFFFF0000u;
        mb[i] = __float_as_uint(v[i] - __uint_as_float(hb[i])) + 0x8000u;
    }
    h = make_uint2(__byte_perm(hb[0], hb[1], 0x7632), __byte_perm(hb[2], hb[3], 0x7632));
    m = make_uint2(__byte_perm(mb[0], mb[1], 0x7632), __byte_perm(mb[2], mb[3], 0x7632));
}

// out = act(scale*y + shift + R)
template <bool VEC>
__global__ void __launch_bounds__(256) bn_apply_kernel(const float* y, const float* scale, const float* shift, int res_mode,
                                                       const float* res, const float* scale2, const float* shift2, int relu,
                                                       float* out, unsigned* mask_bits, RowMap m, long long rows, unsigned short* split = nullptr) {
    constexpr int W = VEC ? 4 : 1;
    const int cq = m.channels / W;
    const long long total = rows * cq;
    // the trip count is uniform per warp (mask words are assembled with full-warp shuffles); lanes past the end idle
    for (long long idx0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); idx0 < total; idx0 += (long long)gridDim.x * blockDim.x) {
        const long long idx = idx0 + (threadIdx.x & 31);
        const bool live = idx < total;
        unsigned nib = 0u;
        if (live) {
        const long long r = idx / cq;
        const int c = (int)(idx - r * cq) * W;
        const long long off = m.row_offset(r) + c;
        if (VEC) {
            float4 v = __ldg(reinterpret_cast<const float4*>(y + off));
            const float4 sc = *reinterpret_cast<const float4*>(scale + c), sh = *reinterpret_cast<const float4*>(shift + c);
            float4 o = make_float4(fmaf(v.x, sc.x, sh.x), fmaf(v.y, sc.y, sh.y), fmaf(v.z, sc.z, sh.z), fmaf(v.w, sc.w, sh.w));
            if (res_mode == AGCN_RES_TENSOR) {
                float4 q = __ldg(reinterpret_cast<const float4*>(res + off));
                o.x += q.x; o.y += q.y; o.z += q.z; o.w += q.w;
            } else if (res_mode == AGCN_RES_AFFINE) {
                float4 q = __ldg(reinterpret_cast<const float4*>(res + off));
                const float4 s2 = *reinterpret_cast<const float4*>(scale2 + c), h2 = *reinterpret_cast<const float4*>(shift2 + c);
                o.x += fmaf(q.x, s2.x, h2.x); o.y += fmaf(q.y, s2.y, h2.y); o.z += fmaf(q.z, s2.z, h2.z); o.w += fmaf(q.w, s2.w, h2.w);
            }
            if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
            *reinterpret_cast<float4*>(out + off) = o;
            if (split != nullptr) {          // the same values as bf16 pieces [2][rows][channels] (contiguous rows only)
                const float ov[4] = {o.x, o.y, o.z, o.w};
                uint2 h, mm;
                bf16_pieces4(ov, h, mm);
                *reinterpret_cast<uint2*>(split + off) = h;
                *reinterpret_cast<uint2*>(split + rows * m.channels + off) = mm;
            }
            nib = (o.x > 0.f ? 1u : 0u) | (o.y > 0.f ? 2u : 0u) | (o.z > 0.f ? 4u : 0u) | (o.w > 0.f ? 8u : 0u);
        } else {
            float o = fmaf(__ldg(y + off), scale[c], shift[c]);
            if (res_mode == AGCN_RES_TENSOR) o += __ldg(res + off);
            else if (res_mode == AGCN_RES_AFFINE) o += fmaf(__ldg(res + off), scale2[c], shift2[c]);
            if (relu) o = fmaxf(o, 0.f);
            out[off] = o;
        }
        }
        if (VEC && mask_bits != nullptr) {
            // eight consecutive lanes hold the 32 bits of one word (element offset = 4 * idx for contiguous rows)
            unsigned wbits = nib << (4u * (threadIdx.x & 7));
            wbits |= __shfl_xor_sync(0xffffffffu, wbits, 1);
            wbits |= __shfl_xor_sync(0xffffffffu, wbits, 2);
            wbits |= __shfl_xor_sync(0xffffffffu, wbits, 4);
            if (live && (threadIdx.x & 7) == 0) mask_bits[idx >> 3] = wbits;
        }
    }
}

// Fused tail of the model (mmargcn/agcn.py:135-136 of the last unit + :194-196): out = relu(scale*y + shift + R) is NOT written; the
// kernel leaves its ReLU mask (one bit per element, for the backward) and the per-group column sums of out.  grid = (parts, groups):
// block (p, g) walks a contiguous slice of the rows of group g; thread = (channel quad, row lane) like colsum_vec_kernel, so eight
// consecutive lanes own the 32 bits of one mask word.  part[(g * parts + p)][channels]; pool_finalize_kernel adds the parts in order.
__global__ void __launch_bounds__(256) bn_apply_pool_kernel(const float* y, const float* scale, const float* shift, int res_mode,
                                                            const float* res, const float* scale2, const float* shift2,
                                                            unsigned* mask_bits, float* part, int rows_per_group, int C) {
    extern __shared__ __align__(16) float smp[];   // [lanes_r][C]
    const int cq = C >> 2;
    const int lanes_r = 256 / cq;
    const int q = threadIdx.x % cq, rl = threadIdx.x / cq;
    const int P = gridDim.x, g = blockIdx.y;
    const int per = (rows_per_group + P - 1) / P;
    const int r0 = blockIdx.x * per;
    int r1 = r0 + per; if (r1 > rows_per_group) r1 = rows_per_group;
    const float4 sc = *reinterpret_cast<const float4*>(scale + q * 4), sh = *reinterpret_cast<const float4*>(shift + q * 4);
    float4 s2 = make_float4(0.f, 0.f, 0.f, 0.f), h2 = s2;
    if (res_mode == AGCN_RES_AFFINE) { s2 = *reinterpret_cast<const float4*>(scale2 + q * 4); h2 = *reinterpret_cast<const float4*>(shift2 + q * 4); }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    // uniform trip count per warp: the mask word is assembled with full-warp shuffles
    for (int rb = r0; rb < r1; rb += lanes_r) {
        const int r = rb + rl;
        const bool live = r < r1;
        unsigned nib = 0u;
        const long long off = ((long long)g * rows_per_group + (live ? r : r0)) * C + q * 4;
        if (live) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(y + off));
            float4 o = make_float4(fmaf(v.x, sc.x, sh.x), fmaf(v.y, sc.y, sh.y), fmaf(v.z, sc.z, sh.z), fmaf(v.w, sc.w, sh.w));
            if (res_mode == AGCN_RES_TENSOR) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(res + off));
                o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w;
            } else if (res_mode == AGCN_RES_AFFINE) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(res + off));
                o.x += fmaf(t.x, s2.x, h2.x); o.y += fmaf(t.y, s2.y, h2.y); o.z += fmaf(t.z, s2.z, h2.z); o.w += fmaf(t.w, s2.w, h2.w);
            }
            o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
            acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
            nib = (o.x > 0.f ? 1u : 0u) | (o.y > 0.f ? 2u : 0u) | (o.z > 0.f ? 4u : 0u) | (o.w > 0.f ? 8u : 0u);
        }
        unsigned wbits = nib << (4u * (threadIdx.x & 7));
        wbits |= __shfl_xor_sync(0xffffffffu, wbits, 1);
        wbits |= __shfl_xor_sync(0xffffffffu, wbits, 2);
        wbits |= __shfl_xor_sync(0xffffffffu, wbits, 4);
        if (live && (threadIdx.x & 7) == 0) mask_bits[off >> 5] = wbits;
    }
    *reinterpret_cast<float4*>(smp + (size_t)rl * C + q * 4) = acc;
    __syncthreads();
    if (rl == 0) {
        float4 t = acc;
        for (int i = 1; i < lanes_r; ++i) {
            const float4 u = *reinterpret_cast<const float4*>(smp + (size_t)i * C + q * 4);
            t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
        }
        *reinterpret_cast<float4*>(part + ((size_t)g * P + blockIdx.x) * C + q * 4) = t;
    }
}

__global__ void pool_finalize_kernel(const float* part, float* pooled, int P, int C, int groups, float inv_rows) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= groups * C) return;
    const int g = idx / C, c = idx - g * C;
    float s = 0.f;
    for (int p = 0; p < P; ++p) s += part[((size_t)g * P + p) * C + c];
    pooled[idx] = s * inv_rows;
}

// coef[0][c] = gamma*invstd, coef[1][c] = s1/m, coef[2][c] = s2/m * invstd, coef[3][c] = mean;  dgamma = s2, dbeta = s1.
// frozen: mean / invstd are constants (eval-mode BatchNorm on its running statistics), so dy = gamma*invstd*g: coef[1] = coef[2] = 0.
__global__ void __launch_bounds__(256) bn_bwd_finalize_kernel(const float* part, int P, int C, double count, const float* gamma,
                                       const float* mean, const float* invstd, float* dgamma, float* dbeta, float* coef, int frozen) {
    const int c = blockIdx.x * kFinCh + threadIdx.x % kFinCh;
    double s1, s2;
    reduce_partials(part, P, C, c, s1, s2);
    if (c >= C || threadIdx.x >= kFinCh) return;
    if (dbeta) dbeta[c] = (float)s1;
    if (dgamma) dgamma[c] = (float)s2;
    const float is = invstd[c];
    coef[0 * C + c] = (gamma ? gamma[c] : 1.f) * is;
    coef[1 * C + c] = frozen ? 0.f : (float)(s1 / count);
    coef[2 * C + c] = frozen ? 0.f : (float)(s2 / count) * is;
    coef[3 * C + c] = mean[c];
}

template <bool VEC>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const float* dout, const float* mask, const unsigned* mask_bits, const float* y,
                                                           const float* coef, float* dy, float* dres, int dres_acc, RowMap m, long long rows,
                                                           int bcast_rows = 0, float bcast_scale = 1.f, unsigned short* dy_split = nullptr) {
    constexpr int W = VEC ? 4 : 1;
    const int C = m.channels;
    const int cq = C / W;
    const long long total = rows * cq;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / cq;
        const int c = (int)(idx - r * cq) * W;
        const long long off = m.row_offset(r) + c;
        float g[4] = {0.f, 0.f, 0.f, 0.f}, yv[4] = {0.f, 0.f, 0.f, 0.f}, mk[4] = {1.f, 1.f, 1.f, 1.f};
        if constexpr (VEC) {
            const float4 a = bcast_rows > 0 ? __ldg(reinterpret_cast<const float4*>(dout + (r / bcast_rows) * C + c))
                                            : __ldg(reinterpret_cast<const float4*>(dout + off));
            g[0] = a.x * bcast_scale; g[1] = a.y * bcast_scale; g[2] = a.z * bcast_scale; g[3] = a.w * bcast_scale;
            if (mask_bits) {
                const unsigned nib = mask_nibble(mask_bits, off);
                mk[0] = (float)(nib & 1u); mk[1] = (float)((nib >> 1) & 1u); mk[2] = (float)((nib >> 2) & 1u); mk[3] = (float)((nib >> 3) & 1u);
            } else if (mask) {
                const float4 k = __ldg(reinterpret_cast<const float4*>(mask + off));
                mk[0] = k.x; mk[1] = k.y; mk[2] = k.z; mk[3] = k.w;
            }
            if (dy) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(y + off));
                yv[0] = b.x; yv[1] = b.y; yv[2] = b.z; yv[3] = b.w;
            }
        } else {
            g[0] = __ldg(dout + off);
            if (mask) mk[0] = __ldg(mask + off);
            if (dy) yv[0] = __ldg(y + off);
        }
        float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int e = 0; e < W; ++e) {
            if (!(mk[e] > 0.f)) g[e] = 0.f;
            if (dy) o[e] = coef[c + e] * (g[e] - coef[C + c + e] - (yv[e] - coef[3 * C + c + e]) * coef[2 * C + c + e]);
        }
        if constexpr (VEC) {
            if (dy) *reinterpret_cast<float4*>(dy + off) = make_float4(o[0], o[1], o[2], o[3]);
            if (dy && dy_split != nullptr) {      // dy once more as bf16 pieces for agcn_conv_wgrad_presplit (contiguous rows only)
                uint2 h, mm;
                bf16_pieces4(o, h, mm);
                *reinterpret_cast<uint2*>(dy_split + off) = h;
                *reinterpret_cast<uint2*>(dy_split + rows * C + off) = mm;
            }
            if (dres) {
                float4 q = make_float4(g[0], g[1], g[2], g[3]);
                if (dres_acc) {
                    const float4 old = *reinterpret_cast<const float4*>(dres + off);
                    q.x += old.x; q.y += old.y; q.z += old.z; q.w += old.w;
                }
                *reinterpret_cast<float4*>(dres + off) = q;
            }
        } else {
            if (dy) dy[off] = o[0];
            if (dres) dres[off] = dres_acc ? dres[off] + g[0] : g[0];
        }
    }
}

// ---- two BatchNorm backwards that share their upstream gradient (the gcn half's bn and down.1 both feed the ReLU of agcn.py:113-115,
// the temporal BatchNorm and the residual branch's both feed the one of :135-136): g = dout * mask is read ONCE per pass for both,
// 8 plane passes instead of 10.  Bit-mask form, contiguous rows, vectorised layout only.
__global__ void __launch_bounds__(256) colsum_dual_kernel(const float* ya, const float* yb, const float* dout, const unsigned* mask_bits,
                                                          const float* mean_a, const float* invstd_a, const float* mean_b, const float* invstd_b,
                                                          int channels, long long rows, float* part_a, float* part_b) {
    extern __shared__ __align__(16) float smv[];   // [4][lanes_r][channels]
    const int cq = channels >> 2;
    const int lanes_r = 256 / cq;
    const int q = threadIdx.x % cq, rl = threadIdx.x / cq;
    const int P = gridDim.x;
    const long long per = (rows + P - 1) / P;
    const long long r0 = (long long)blockIdx.x * per;
    long long r1 = r0 + per; if (r1 > rows) r1 = rows;
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), sa = s0, sb = s0;      // sum g (shared by both), sum g xhat_a, sum g xhat_b
    const float4 mua = *reinterpret_cast<const float4*>(mean_a + q * 4), isa = *reinterpret_cast<const float4*>(invstd_a + q * 4);
    const float4 mub = *reinterpret_cast<const float4*>(mean_b + q * 4), isb = *reinterpret_cast<const float4*>(invstd_b + q * 4);
    auto body = [&](float4 g, unsigned nib, const float4& va, const float4& vb) {
        if (!(nib & 1u)) g.x = 0.f;
        if (!(nib & 2u)) g.y = 0.f;
        if (!(nib & 4u)) g.z = 0.f;
        if (!(nib & 8u)) g.w = 0.f;
        s0.x += g.x; s0.y += g.y; s0.z += g.z; s0.w += g.w;
        sa.x = fmaf(g.x, (va.x - mua.x) * isa.x, sa.x); sa.y = fmaf(g.y, (va.y - mua.y) * isa.y, sa.y);
        sa.z = fmaf(g.z, (va.z - mua.z) * isa.z, sa.z); sa.w = fmaf(g.w, (va.w - mua.w) * isa.w, sa.w);
        sb.x = fmaf(g.x, (vb.x - mub.x) * isb.x, sb.x); sb.y = fmaf(g.y, (vb.y - mub.y) * isb.y, sb.y);
        sb.z = fmaf(g.z, (vb.z - mub.z) * isb.z, sb.z); sb.w = fmaf(g.w, (vb.w - mub.w) * isb.w, sb.w);
    };
    long long r = r0 + rl;
    for (; r + lanes_r < r1; r += 2LL * lanes_r) {          // two rows per trip, all six loads first (see colsum_vec_kernel)
        const long long o0 = r * channels + q * 4, o1 = (r + lanes_r) * channels + q * 4;
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(dout + o0)), g1 = __ldg(reinterpret_cast<const float4*>(dout + o1));
        const float4 a0 = __ldg(reinterpret_cast<const float4*>(ya + o0)), a1 = __ldg(reinterpret_cast<const float4*>(ya + o1));
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(yb + o0)), b1 = __ldg(reinterpret_cast<const float4*>(yb + o1));
        const unsigned n0 = mask_nibble(mask_bits, o0), n1 = mask_nibble(mask_bits, o1);
        body(g0, n0, a0, b0);
        body(g1, n1, a1, b1);
    }
    for (; r < r1; r += lanes_r) {
        const long long o0 = r * channels + q * 4;
        body(__ldg(reinterpret_cast<const float4*>(dout + o0)), mask_nibble(mask_bits, o0),
             __ldg(reinterpret_cast<const float4*>(ya + o0)), __ldg(reinterpret_cast<const float4*>(yb + o0)));
    }
    float4* a = reinterpret_cast<float4*>(smv);
    a[(0 * lanes_r + rl) * cq + q] = s0;
    a[(1 * lanes_r + rl) * cq + q] = sa;
    a[(2 * lanes_r + rl) * cq + q] = sb;
    __syncthreads();
    for (int o = threadIdx.x; o < 3 * channels; o += 256) {
        const int which = o / channels, c = o % channels;
        float acc = 0.f;
        for (int i = 0; i < lanes_r; ++i) acc += smv[(which * lanes_r + i) * channels + c];
        if (which == 0) {
            part_a[((long long)blockIdx.x * 2 + 0) * channels + c] = acc;
            part_b[((long long)blockIdx.x * 2 + 0) * channels + c] = acc;
        } else if (which == 1) {
            part_a[((long long)blockIdx.x * 2 + 1) * channels + c] = acc;
        } else {
            part_b[((long long)blockIdx.x * 2 + 1) * channels + c] = acc;
        }
    }
}

__global__ void __launch_bounds__(256) bn_bwd_apply_dual_kernel(const float* dout, const unsigned* mask_bits, const float* ya, const float* yb,
                                                                const float* coef_a, const float* coef_b, float* dya, float* dyb,
                                                                unsigned short* dya_split, int C, long long rows) {
    const int cq = C / 4;
    const long long total = rows * cq;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / cq;
        const int c = (int)(idx - r * cq) * 4;
        const long long off = r * C + c;
        const float4 gq = __ldg(reinterpret_cast<const float4*>(dout + off));
        const float4 aq = __ldg(reinterpret_cast<const float4*>(ya + off));
        const float4 bq = __ldg(reinterpret_cast<const float4*>(yb + off));
        const unsigned nib = mask_nibble(mask_bits, off);
        float g[4] = {gq.x, gq.y, gq.z, gq.w};
        const float av[4] = {aq.x, aq.y, aq.z, aq.w}, bv[4] = {bq.x, bq.y, bq.z, bq.w};
        float oa[4], ob[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (!((nib >> e) & 1u)) g[e] = 0.f;
            oa[e] = coef_a[c + e] * (g[e] - coef_a[C + c + e] - (av[e] - coef_a[3 * C + c + e]) * coef_a[2 * C + c + e]);
            ob[e] = coef_b[c + e] * (g[e] - coef_b[C + c + e] - (bv[e] - coef_b[3 * C + c + e]) * coef_b[2 * C + c + e]);
        }
        *reinterpret_cast<float4*>(dya + off) = make_float4(oa[0], oa[1], oa[2], oa[3]);
        *reinterpret_cast<float4*>(dyb + off) = make_float4(ob[0], ob[1], ob[2], ob[3]);
        if (dya_split != nullptr) {
            uint2 h, mm;
            bf16_pieces4(oa, h, mm);
            *reinterpret_cast<uint2*>(dya_split + off) = h;
            *reinterpret_cast<uint2*>(dya_split + rows * C + off) = mm;
        }
    }
}

// pooling: grid = (groups, column strips of 32); block = 32 x 8
__global__ void __launch_bounds__(256) pool_fwd_kernel(const float* x, float* out, int rows_per_group, int C) {
    __shared__ float sm[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.y * 32 + tx;
    const float* base = x + (long long)blockIdx.x * rows_per_group * C;
    float s = 0.f;
    if (c < C)
        for (int r = ty; r < rows_per_group; r += 8) s += __ldg(base + (long long)r * C + c);
    sm[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && c < C) {
        float a = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) a += sm[i][tx];
        out[(long long)blockIdx.x * C + c] = a / (float)rows_per_group;
    }
}

__global__ void pool_bwd_kernel(const float* dout, float* dx, int rows_per_group, int C, long long total) {
    const float inv = 1.f / (float)rows_per_group;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % C);
        const long long g = idx / ((long long)rows_per_group * C);
        dx[idx] = dout[g * C + c] * inv;
    }
}

static bool vec_ok(const RowMap& m, std::initializer_list<const void*> ptrs) {
    if (m.channels % 4) return false;
    if (m.outer != 1 && (m.outer_stride % 4)) return false;
    for (const void* p : ptrs) if (p != nullptr && !aligned16(p)) return false;
    return true;
}

static bool colsum_vec_shape(const RowMap& m) {
    const int cq = m.channels / 4;
    return m.channels % 4 == 0 && cq <= 256 && (256 % cq) == 0 && m.channels <= 1024;
}

template <int MODE>
static int launch_colsum(const float* x, const float* dout, const float* mask, const float* mean, const float* invstd,
                         const RowMap& m, long long rows, float* part, int P, cudaStream_t s, const unsigned* mask_bits = nullptr,
                         int bcast_rows = 0, float bcast_scale = 1.f) {
    const int cq = m.channels / 4;
    const bool vec = vec_ok(m, {x, dout, mask, mean, invstd}) && colsum_vec_shape(m);
    if ((mask_bits != nullptr || bcast_rows > 0) && !vec) return fail(AGCN_ERR_UNSUPPORTED, "bn column sums: a bit mask needs the vectorised layout");
    if (vec) {
        const int lanes_r = 256 / cq;
        size_t smem = (size_t)2 * lanes_r * m.channels * sizeof(float);
        colsum_vec_kernel<MODE><<<P, 256, smem, s>>>(x, dout, mask, mask_bits, mean, invstd, m, rows, part, bcast_rows, bcast_scale);
    } else {
        dim3 grid((unsigned)P, (unsigned)ceil_div(m.channels, 32));
        colsum_strip_kernel<MODE><<<grid, 256, 0, s>>>(x, dout, mask, mean, invstd, m, rows, part);
    }
    return check_launch("bn column sums");
}

static int elementwise_blocks(long long work_items) {
    long long b = (work_items + 255) / 256;
    const long long cap = (long long)kNumSMs * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

}  // namespace agcn

using namespace agcn;

extern "C" AGCN_API size_t agcn_bn_workspace_bytes(int channels) {
    if (channels <= 0) return 0;
    // partial sums [kMaxPartials][2][C] followed by the backward coefficients [4][C]
    return ((size_t)kMaxPartials * 2 + 4) * (size_t)channels * sizeof(float);
}

static int check_map(const char* who, int outer, int inner, long long outer_stride, int channels) {
    AGCN_REQUIRE(outer > 0 && inner > 0 && channels > 0, AGCN_ERR_BAD_SHAPE, "%s: bad shape outer=%d inner=%d channels=%d", who, outer, inner, channels);
    AGCN_REQUIRE(outer == 1 || outer_stride >= (long long)inner * channels, AGCN_ERR_BAD_SHAPE, "%s: outer_stride too small", who);
    return AGCN_OK;
}

extern "C" AGCN_API int agcn_bn_stats(const float* x, int outer, int inner, long long outer_stride, int channels,
                             const float* gamma, const float* beta, float* running_mean, float* running_var,
                             long long* num_batches_tracked, float momentum, float eps, int training,
                             float* scale, float* shift, float* save_mean, float* save_invstd,
                             void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_map("agcn_bn_stats", outer, inner, outer_stride, channels);
    if (rc) return rc;
    AGCN_REQUIRE(scale && shift, AGCN_ERR_NULL, "agcn_bn_stats: scale/shift are required");
    AGCN_REQUIRE(training || (running_mean && running_var), AGCN_ERR_NULL, "agcn_bn_stats: eval mode needs running statistics");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    RowMap m{outer, inner, outer_stride, channels};
    const long long rows = (long long)outer * inner;
    int P = 0;
    float* part = static_cast<float*>(workspace);
    if (training) {
        AGCN_REQUIRE(x && workspace, AGCN_ERR_NULL, "agcn_bn_stats: null pointer");
        AGCN_REQUIRE(workspace_bytes >= agcn_bn_workspace_bytes(channels), AGCN_ERR_WORKSPACE, "agcn_bn_stats: workspace too small");
        P = num_partials(rows);
        // pivot of the shifted sums: the first row of x (any value near the channel's mean removes the cancellation)
        rc = launch_colsum<0>(x, nullptr, nullptr, x, nullptr, m, rows, part, P, s);
        if (rc) return rc;
    }
    bn_finalize_kernel<<<ceil_div(channels, kFinCh), kFinCh * kFinLanes, 0, s>>>(part, P, channels, (double)rows, gamma, beta, running_mean, running_var,
                                                              num_batches_tracked, momentum, eps, training, scale, shift, save_mean, save_invstd,
                                                              training ? x : nullptr, 0);
    return check_launch("agcn_bn_stats(finalize)");
}

extern "C" AGCN_API int agcn_bn_finalize(const float* part, int nparts, long long rows, int channels,
                                const float* gamma, const float* beta, float* running_mean, float* running_var,
                                long long* num_batches_tracked, float momentum, float eps,
                                float* scale, float* shift, float* save_mean, float* save_invstd, void* stream) {
    AGCN_REQUIRE(part && scale && shift, AGCN_ERR_NULL, "agcn_bn_finalize: null pointer");
    AGCN_REQUIRE(nparts > 0 && rows > 0 && channels > 0, AGCN_ERR_BAD_SHAPE, "agcn_bn_finalize: bad shape nparts=%d rows=%lld channels=%d",
                 nparts, rows, channels);
    bn_finalize_kernel<<<ceil_div(channels, kFinCh), kFinCh * kFinLanes, 0, static_cast<cudaStream_t>(stream)>>>(
        part, nparts, channels, (double)rows, gamma, beta, running_mean, running_var, num_batches_tracked, momentum, eps, 1,
        scale, shift, save_mean, save_invstd, nullptr, 1);
    return check_launch("agcn_bn_finalize");
}

extern "C" AGCN_API size_t agcn_bn_mask_words(int outer, int inner, int channels) {
    // one bit per element of a CONTIGUOUS [rows][channels] tensor; only layouts both the writer (agcn_bn_apply) and the
    // reader (agcn_bn_bwd) vectorise are supported -- 0 otherwise (use the fp32 tensor as the mask then)
    if (outer != 1 || inner <= 0 || channels <= 0) return 0;
    RowMap m{1, inner, 0, channels};
    if (!colsum_vec_shape(m)) return 0;
    return (size_t)(((long long)inner * channels + 31) / 32);
}

// mask_bits / out_split (NULL: not written): the ReLU mask as one bit per element and `out` as bf16 pieces [2][inner][channels]
// (plane 0 = h = bf16(out), plane 1 = m = bf16(out - h)), the operand format of agcn_conv_wgrad_presplit -- the weight gradient of
// the convolution that consumes `out` then needs no conversion pass of its own.
extern "C" AGCN_API int agcn_bn_apply(const float* y, const float* scale, const float* shift,
                                      int res_mode, const float* res, const float* scale2, const float* shift2,
                                      int relu, float* out, unsigned* mask_bits, void* out_split,
                                      int outer, int inner, long long outer_stride, int channels, void* stream) {
    int rc = check_map("agcn_bn_apply", outer, inner, outer_stride, channels);
    if (rc) return rc;
    AGCN_REQUIRE(y && scale && shift && out, AGCN_ERR_NULL, "agcn_bn_apply: null pointer");
    AGCN_REQUIRE(res_mode == AGCN_RES_NONE || res, AGCN_ERR_NULL, "agcn_bn_apply: residual tensor missing");
    AGCN_REQUIRE(res_mode != AGCN_RES_AFFINE || (scale2 && shift2), AGCN_ERR_NULL, "agcn_bn_apply: scale2/shift2 missing");
    AGCN_REQUIRE(res_mode >= 0 && res_mode <= 2, AGCN_ERR_UNSUPPORTED, "agcn_bn_apply: res_mode %d", res_mode);
    RowMap m{outer, inner, outer_stride, channels};
    const long long rows = (long long)outer * inner;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned short* split = static_cast<unsigned short*>(out_split);
    const bool vec = vec_ok(m, {y, scale, shift, res, scale2, shift2, out});
    if (mask_bits != nullptr)
        AGCN_REQUIRE(vec && agcn_bn_mask_words(outer, inner, channels) > 0, AGCN_ERR_UNSUPPORTED,
                     "agcn_bn_apply: mask_bits: layout not supported (agcn_bn_mask_words returned 0)");
    if (split != nullptr)
        AGCN_REQUIRE(vec && outer == 1 && aligned16(split), AGCN_ERR_UNSUPPORTED, "agcn_bn_apply: out_split needs a contiguous, vectorisable layout");
    if (vec)
        bn_apply_kernel<true><<<elementwise_blocks(rows * (channels / 4)), 256, 0, s>>>(y, scale, shift, res_mode, res, scale2, shift2, relu, out, mask_bits, m, rows, split);
    else
        bn_apply_kernel<false><<<elementwise_blocks(rows * channels), 256, 0, s>>>(y, scale, shift, res_mode, res, scale2, shift2, relu, out, nullptr, m, rows);
    return check_launch("agcn_bn_apply");
}

// phase 0: the whole backward.  Synchronised BatchNorm (statistics over all ranks) splits it around the caller's all-reduce:
// phase 1 = column sums only (dbeta = sum g, dgamma = sum g xhat of THIS rank's rows), phase 2 = the apply pass from
// global_sums [2][C] = (sum g | sum g xhat) over all ranks and the global row count.
// pool_rows > 0: dout is the gradient of the fused mean pool, [inner / pool_rows][C], broadcast over the rows of each group.
extern "C" AGCN_API int agcn_bn_bwd(const float* dout, const float* mask_out, const unsigned* mask_bits, const float* y,
                                    const float* save_mean, const float* save_invstd, const float* gamma,
                                    float* dy, void* dy_split, float* dgamma, float* dbeta, float* dres, int dres_accumulate,
                                    int frozen_stats, int outer, int inner, long long outer_stride, int channels, int pool_rows,
                                    int phase, const float* global_sums, double global_rows,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_map("agcn_bn_bwd", outer, inner, outer_stride, channels);
    if (rc) return rc;
    AGCN_REQUIRE(phase >= 0 && phase <= 2, AGCN_ERR_UNSUPPORTED, "agcn_bn_bwd: phase %d", phase);
    AGCN_REQUIRE(!frozen_stats || (pool_rows == 0 && phase == 0), AGCN_ERR_UNSUPPORTED,
                 "agcn_bn_bwd: frozen statistics take neither a pooled gradient nor the synchronised phases");
    AGCN_REQUIRE(!(mask_out && mask_bits), AGCN_ERR_UNSUPPORTED, "agcn_bn_bwd: mask_out and mask_bits are alternatives, not both");
    AGCN_REQUIRE(phase != 1 || (dgamma && dbeta), AGCN_ERR_NULL, "agcn_bn_bwd: phase 1 writes dgamma / dbeta");
    AGCN_REQUIRE(!dy_split || dy, AGCN_ERR_NULL, "agcn_bn_bwd: dy_split needs dy");
    AGCN_REQUIRE(pool_rows >= 0 && (pool_rows == 0 || (outer == 1 && inner % pool_rows == 0)), AGCN_ERR_BAD_SHAPE, "agcn_bn_bwd: bad pooled shape");
    AGCN_REQUIRE(pool_rows == 0 || mask_bits, AGCN_ERR_NULL, "agcn_bn_bwd: a pooled gradient needs mask_bits");
    AGCN_REQUIRE(dout && y && save_mean && save_invstd && workspace, AGCN_ERR_NULL, "agcn_bn_bwd: null pointer");
    AGCN_REQUIRE(workspace_bytes >= agcn_bn_workspace_bytes(channels), AGCN_ERR_WORKSPACE, "agcn_bn_bwd: workspace too small");
    RowMap m{outer, inner, outer_stride, channels};
    const long long rows = (long long)outer * inner;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float* part = static_cast<float*>(workspace);
    float* coef = part + (size_t)kMaxPartials * 2 * channels;
    unsigned short* split = static_cast<unsigned short*>(dy_split);
    const int P = num_partials(rows);
    if (mask_bits != nullptr)
        AGCN_REQUIRE(agcn_bn_mask_words(outer, inner, channels) > 0 && vec_ok(m, {dout, y, dy, dres, workspace}), AGCN_ERR_UNSUPPORTED,
                     "agcn_bn_bwd: mask_bits: layout not supported (agcn_bn_mask_words returned 0)");
    const float bcast_scale = pool_rows > 0 ? 1.f / (float)pool_rows : 1.f;
    if (phase == 2) {
        AGCN_REQUIRE(global_sums && global_rows >= (double)rows, AGCN_ERR_NULL, "agcn_bn_bwd: phase 2 needs the all-reduced sums and the global row count");
        bn_bwd_finalize_kernel<<<ceil_div(channels, kFinCh), kFinCh * kFinLanes, 0, s>>>(global_sums, 1, channels, global_rows, gamma, save_mean, save_invstd,
                                                                                         nullptr, nullptr, coef, frozen_stats);
    } else {
        rc = launch_colsum<1>(y, dout, mask_out, save_mean, save_invstd, m, rows, part, P, s, mask_bits, pool_rows, bcast_scale);
        if (rc) return rc;
        bn_bwd_finalize_kernel<<<ceil_div(channels, kFinCh), kFinCh * kFinLanes, 0, s>>>(part, P, channels, (double)rows, gamma, save_mean, save_invstd, dgamma, dbeta, coef, frozen_stats);
    }
    rc = check_launch("agcn_bn_bwd(finalize)");
    if (rc) return rc;
    if (phase == 1 || (dy == nullptr && dres == nullptr)) return AGCN_OK;
    if (split != nullptr)
        AGCN_REQUIRE(outer == 1 && aligned16(split) && vec_ok(m, {dout, mask_out, y, dy, dres, coef}), AGCN_ERR_UNSUPPORTED,
                     "agcn_bn_bwd: dy_split needs a contiguous, vectorisable layout");
    if (vec_ok(m, {dout, mask_out, y, dy, dres, coef}))
        bn_bwd_apply_kernel<true><<<elementwise_blocks(rows * (channels / 4)), 256, 0, s>>>(dout, mask_out, mask_bits, y, coef, dy, dres, dres_accumulate, m, rows,
                                                                                            pool_rows, bcast_scale, split);
    else
        bn_bwd_apply_kernel<false><<<elementwise_blocks(rows * channels), 256, 0, s>>>(dout, mask_out, nullptr, y, coef, dy, dres, dres_accumulate, m, rows);
    return check_launch("agcn_bn_bwd(apply)");
}

// Two BatchNorm backwards over the same masked upstream gradient in one pair of passes (see colsum_dual_kernel): BatchNorm A = (y_a,
// mean_a, invstd_a, gamma_a) -> dy_a (+ dy_a_split, optional bf16 pieces), dgamma_a, dbeta_a; BatchNorm B likewise without pieces.
// workspace: 2 x agcn_bn_workspace_bytes(channels).  AGCN_ERR_UNSUPPORTED (quiet) when the layout has no bit mask (agcn_bn_mask_words == 0).
extern "C" AGCN_API int agcn_bn_bwd_bits_dual(const float* dout, const unsigned* mask_bits,
                                              const float* y_a, const float* mean_a, const float* invstd_a, const float* gamma_a,
                                              float* dy_a, void* dy_a_split, float* dgamma_a, float* dbeta_a,
                                              const float* y_b, const float* mean_b, const float* invstd_b, const float* gamma_b,
                                              float* dy_b, float* dgamma_b, float* dbeta_b,
                                              int frozen_stats, int inner, int channels, void* workspace, size_t workspace_bytes, void* stream) {
    AGCN_REQUIRE(dout && mask_bits && y_a && mean_a && invstd_a && dy_a && y_b && mean_b && invstd_b && dy_b && workspace, AGCN_ERR_NULL,
                 "agcn_bn_bwd_bits_dual: null pointer");
    AGCN_REQUIRE(inner > 0 && channels > 0, AGCN_ERR_BAD_SHAPE, "agcn_bn_bwd_bits_dual: bad shape inner=%d channels=%d", inner, channels);
    const size_t one = agcn_bn_workspace_bytes(channels);
    AGCN_REQUIRE(workspace_bytes >= 2 * one, AGCN_ERR_WORKSPACE, "agcn_bn_bwd_bits_dual: workspace too small");
    RowMap m{1, inner, 0, channels};
    if (agcn_bn_mask_words(1, inner, channels) == 0 ||
        !vec_ok(m, {dout, y_a, y_b, dy_a, dy_b, mean_a, invstd_a, mean_b, invstd_b, workspace, dy_a_split}))
        return AGCN_ERR_UNSUPPORTED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const long long rows = inner;
    const int P = num_partials(rows);
    float* part_a = static_cast<float*>(workspace);
    float* coef_a = part_a + (size_t)kMaxPartials * 2 * channels;
    float* part_b = reinterpret_cast<float*>(static_cast<char*>(workspace) + one);
    float* coef_b = part_b + (size_t)kMaxPartials * 2 * channels;
    const int cq = channels / 4;
    const size_t smem = (size_t)3 * (256 / cq) * channels * sizeof(float);
    colsum_dual_kernel<<<P, 256, smem, s>>>(y_a, y_b, dout, mask_bits, mean_a, invstd_a, mean_b, invstd_b, channels, rows, part_a, part_b);
    int rc = check_launch("agcn_bn_bwd_bits_dual(sums)");
    if (rc) return rc;
    bn_bwd_finalize_kernel<<<ceil_div(channels, kFinCh), kFinCh * kFinLanes, 0, s>>>(part_a, P, channels, (double)rows, gamma_a, mean_a, invstd_a, dgamma_a, dbeta_a, coef_a, frozen_stats);
    bn_bwd_finalize_kernel<<<ceil_div(channels, kFinCh), kFinCh * kFinLanes, 0, s>>>(part_b, P, channels, (double)rows, gamma_b, mean_b, invstd_b, dgamma_b, dbeta_b, coef_b, frozen_stats);
    rc = check_launch("agcn_bn_bwd_bits_dual(finalize)");
    if (rc) return rc;
    bn_bwd_apply_dual_kernel<<<elementwise_blocks(rows * cq), 256, 0, s>>>(dout, mask_bits, y_a, y_b, coef_a, coef_b, dy_a, dy_b,
                                                                           static_cast<unsigned short*>(dy_a_split), channels, rows);
    return check_launch("agcn_bn_bwd_bits_dual(apply)");
}

// ---- synchronised BatchNorm (statistics over all ranks of a data-parallel group; SURVEY 8e "optional SyncBN mode")
// The collectives stay with the caller (torch.distributed / NCCL); the library provides the two halves either side of them.

// part4 [P][4][C]: per row-partition p the shifted sum | shifted sum of squares | pivot | row count -- the layout agcn_bn_finalize merges
// (the same one the convolution epilogue writes), so the partials of several ranks can simply be concatenated.
__global__ void expand_partials_kernel(const float* part2, const float* x_first_row, int P, int C, long long rows, float* part4) {
    const long long per = (rows + P - 1) / P;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < P * C; idx += gridDim.x * blockDim.x) {
        const int p = idx / C, c = idx - p * C;
        long long n = rows - (long long)p * per;
        n = n < 0 ? 0 : (n > per ? per : n);
        part4[((long long)p * 4 + 0) * C + c] = part2[((long long)p * 2 + 0) * C + c];
        part4[((long long)p * 4 + 1) * C + c] = part2[((long long)p * 2 + 1) * C + c];
        part4[((long long)p * 4 + 2) * C + c] = x_first_row[c];
        part4[((long long)p * 4 + 3) * C + c] = (float)n;
    }
}

extern "C" AGCN_API size_t agcn_bn_stats_partials_bytes(int channels) {
    return channels > 0 ? (size_t)agcn::kMaxPartials * 4 * (size_t)channels * sizeof(float) : 0;
}

extern "C" AGCN_API int agcn_bn_stats_partials(const float* x, int outer, int inner, long long outer_stride, int channels,
                                               float* part, size_t part_bytes, int* nparts,
                                               void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_map("agcn_bn_stats_partials", outer, inner, outer_stride, channels);
    if (rc) return rc;
    AGCN_REQUIRE(x && part && nparts && workspace, AGCN_ERR_NULL, "agcn_bn_stats_partials: null pointer");
    AGCN_REQUIRE(workspace_bytes >= agcn_bn_workspace_bytes(channels), AGCN_ERR_WORKSPACE, "agcn_bn_stats_partials: workspace too small");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    RowMap m{outer, inner, outer_stride, channels};
    const long long rows = (long long)outer * inner;
    const int P = num_partials(rows);
    AGCN_REQUIRE(part_bytes >= (size_t)P * 4 * channels * sizeof(float), AGCN_ERR_WORKSPACE, "agcn_bn_stats_partials: partial buffer too small");
    float* part2 = static_cast<float*>(workspace);
    rc = launch_colsum<0>(x, nullptr, nullptr, x, nullptr, m, rows, part2, P, s);      // pivot = the first row of x
    if (rc) return rc;
    expand_partials_kernel<<<ceil_div(P * channels, 256), 256, 0, s>>>(part2, x, P, channels, rows, part);
    *nparts = P;
    return check_launch("agcn_bn_stats_partials");
}

constexpr int kPoolParts = 8;

extern "C" AGCN_API size_t agcn_bn_apply_pool_workspace_bytes(int groups, int channels) {
    return (groups > 0 && channels > 0) ? (size_t)groups * kPoolParts * channels * sizeof(float) : 0;
}

extern "C" AGCN_API int agcn_bn_apply_pool(const float* y, const float* scale, const float* shift,
                                           int res_mode, const float* res, const float* scale2, const float* shift2,
                                           unsigned* mask_bits, float* pooled, int groups, int rows_per_group, int channels,
                                           void* workspace, size_t workspace_bytes, void* stream) {
    AGCN_REQUIRE(y && scale && shift && mask_bits && pooled && workspace, AGCN_ERR_NULL, "agcn_bn_apply_pool: null pointer");
    AGCN_REQUIRE(groups > 0 && rows_per_group > 0 && channels > 0, AGCN_ERR_BAD_SHAPE, "agcn_bn_apply_pool: bad shape");
    AGCN_REQUIRE(res_mode >= 0 && res_mode <= 2 && (res_mode == AGCN_RES_NONE || res) && (res_mode != AGCN_RES_AFFINE || (scale2 && shift2)),
                 AGCN_ERR_NULL, "agcn_bn_apply_pool: residual operands missing");
    AGCN_REQUIRE(workspace_bytes >= agcn_bn_apply_pool_workspace_bytes(groups, channels), AGCN_ERR_WORKSPACE, "agcn_bn_apply_pool: workspace too small");
    RowMap m{1, groups * rows_per_group, 0, channels};
    AGCN_REQUIRE(agcn_bn_mask_words(1, groups * rows_per_group, channels) > 0 && channels % 32 == 0 &&
                 vec_ok(m, {y, scale, shift, res, scale2, shift2, pooled, workspace}),
                 AGCN_ERR_UNSUPPORTED, "agcn_bn_apply_pool: layout not supported (use agcn_bn_apply + agcn_pool_fwd)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float* part = static_cast<float*>(workspace);
    const int cq = channels / 4;
    const size_t smem = (size_t)(256 / cq) * channels * sizeof(float);
    dim3 grid((unsigned)kPoolParts, (unsigned)groups);
    bn_apply_pool_kernel<<<grid, 256, smem, s>>>(y, scale, shift, res_mode, res, scale2, shift2, mask_bits, part, rows_per_group, channels);
    int rc = check_launch("agcn_bn_apply_pool");
    if (rc) return rc;
    pool_finalize_kernel<<<ceil_div((long long)groups * channels, 256), 256, 0, s>>>(part, pooled, kPoolParts, channels, groups, 1.f / (float)rows_per_group);
    return check_launch("agcn_bn_apply_pool(finalize)");
}

extern "C" AGCN_API int agcn_pool_fwd(const float* x, float* out, int groups, int rows_per_group, int channels, void* stream) {
    AGCN_REQUIRE(x && out, AGCN_ERR_NULL, "agcn_pool_fwd: null pointer");
    AGCN_REQUIRE(groups > 0 && rows_per_group > 0 && channels > 0, AGCN_ERR_BAD_SHAPE, "agcn_pool_fwd: bad shape");
    dim3 grid((unsigned)groups, (unsigned)ceil_div(channels, 32));
    pool_fwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, out, rows_per_group, channels);
    return check_launch("agcn_pool_fwd");
}

extern "C" AGCN_API int agcn_pool_bwd(const float* dout, float* dx, int groups, int rows_per_group, int channels, void* stream) {
    AGCN_REQUIRE(dout && dx, AGCN_ERR_NULL, "agcn_pool_bwd: null pointer");
    AGCN_REQUIRE(groups > 0 && rows_per_group > 0 && channels > 0, AGCN_ERR_BAD_SHAPE, "agcn_pool_bwd: bad shape");
    const long long total = (long long)groups * rows_per_group * channels;
    pool_bwd_kernel<<<elementwise_blocks(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(dout, dx, rows_per_group, channels, total);
    return check_launch("agcn_pool_bwd");
}
