// tcgen05 / TMA tensor-core weight gradient of the implicit GEMM, sm_100a only (the forward / input-gradient contraction
// lives in conv_tc2.cu).
//
//   dw[co][tap][ci] = sum_rows dy[nb][to][v][co] * x[nb][stride*to+tap-pad][v][ci]
//
// Precision.  tcgen05.mma kind::tf32 reads fp32 words from shared memory and uses their upper 19 bits (measured on
// B200: results match an fp64 contraction of TF32-TRUNCATED operands to 1e-6).  SPLIT = false is that single pass
// (AGCN_PREC_TF32).  SPLIT = true is the fp32-parity mode (AGCN_PREC_FP32, "3xTF32"): with hi = rna_tf32(x) (round to
// nearest, so the split is unbiased) and lo = x - hi (exact in fp32), it issues
//   lo_a*hi_b + hi_a*lo_b + hi_a*hi_b  =  a*b - lo_a*lo_b  (relative error ~2^-22 per product)
#include "tc_common.cuh"
#include <stdlib.h>

namespace agcn {
namespace tc {

constexpr int kThreads = 192;               // TMA warp, MMA warp, 4 epilogue warps

constexpr int kWgTransformWarps = 8;                       // 3xTF32 weight gradient: operand-split warps
constexpr int kWgStages = 8;                               // barrier slots of the weight-gradient raw ring
constexpr int kWgBarBytes = 512;
constexpr int kWgThreadsSplit = (6 + kWgTransformWarps) * 32;

struct WgArgs {
    float* ws;
    int nb, t_in, t_out, v, cin, cout, taps, stride, pad;
    int flat, rows_box, rpad, tt, chunks_per_sample;
    long long chunks_total, chunks_per_split;
    int n_tile, n_tiles, m_tiles, stages;
    int pair;          // 1: a tile is two consecutive taps stacked along M (cout <= 64): lanes 0..63 = tap 2j, lanes 64..127 = tap 2j+1
    int tap_tiles;     // taps, or ceil(taps / 2) in pair mode
    int seg_chunks;    // 3xTF32: row chunks per accumulator segment (promoted to fp32 registers in between)
    int blocked;       // 1: tensor maps carry the 32-channel block as its own dimension: ONE TMA box per operand and stage
    int nblk_a;        // blocked: dy channel blocks per box (<= 4; pair mode: 2, loaded twice)
    int pre_ablk, pre_bblk;   // MODE 3: 64-channel blocks per dy / x box (the transaction bytes count whole boxes, out-of-range blocks included)
    int dbg;           // bring-up only (env AGCN_WG_DEBUG): bit 0 skips the operand split, bit 1 skips the MMAs -> wrong results, timing probes
};


// MODE: 0 single-pass TF32, 1 3xTF32, 2 BF16x3.  BF16x3: the TMA boxes are plain-128B-swizzled fp32 blocks of 32 channels; the
// converter warps (one thread per K row) rewrite every PAIR of slots in place as 64 bf16 channels of h (first slot) and of m
// (second slot) -- MN-major 16-bit operands, 64 channels per 128-byte row, 8-row swizzle groups -- and the issuer runs
// h.h + h.m + m.h on kind::f16 with K = 16 rows per MMA.  No lo ring: four 48 KB stages like the TF32 mode.
// MODE 3: BF16x3 on operands that ARRIVE split -- [2][rows][C] bf16 tensors (plane 0 = h, plane 1 = m) written by the kernels that
// produced the activations / gradients (agcn_bn_apply / agcn_bn_bwd with out_split / dy_split).  One 5-D TMA box per operand lands as
// [64-channel block][piece][row][128 B], which IS the slot layout the issuer reads (h in the even slots, m in the odd ones): no
// converter warps, no in-place rewrite -- the kernel is the TF32-mode pipeline with three bf16 MMAs per 16 rows.  In the in-kernel
// conversion (MODE 2) the shared memory moves ~216 KB per 48 KB stage (TMA landing, conversion read + write, operand reads of three
// MMAs), which bounds it at ~200 TFLOP/s; here it moves 120 KB.
template <int MODE>
__global__ void __launch_bounds__((MODE == 1 || MODE == 2) ? kWgThreadsSplit : kThreads, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x,
                const __grid_constant__ CUtensorMap map_dy_m, const __grid_constant__ CUtensorMap map_x_m, WgArgs a) {
    // (map_dy_m / map_x_m: MODE 3 with whole-timestep boxes -- strided / shortened convolutions -- loads the h and the m plane through
    // separate 5-D maps (64 channels, v, t, block, sample), one box per (64-channel block, piece); unused otherwise)
    constexpr bool SPLIT = MODE == 1, PRE = MODE == 3, BF = MODE == 2 || MODE == 3, CONV = MODE != 0;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sub_bytes = (uint32_t)a.rpad * 128u;
    const uint32_t nsub_b = (uint32_t)a.n_tile / 32u;
    const uint32_t nsub_slots = BF ? ((nsub_b + 1u) & ~1u) : nsub_b;      // BF16x3: x slots come in (h, m) pairs
    const uint32_t raw_bytes = (4u + nsub_slots) * sub_bytes;             // one stage of TMA payload (raw, becomes hi / h|m in place)
    const uint32_t lo_ring = smem_base + (uint32_t)a.stages * raw_bytes;  // SPLIT: two slots of lo residuals
    const uint32_t bar_base = lo_ring + (SPLIT ? 2u * raw_bytes : 0u);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (kWgStages + s); };
    auto lo_bar = [&](int s) { return bar_base + 8u * (2 * kWgStages + s); };
    auto lo_empty = [&](int s) { return bar_base + 8u * (3 * kWgStages + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (3 * kWgStages + 2 + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (3 * kWgStages + 4 + s); };
    const uint32_t tmem_slot = bar_base + 8u * (3 * kWgStages + 6);
    constexpr int kCols = CONV ? 512 : 256;                               // parity modes: 2 x 128 segment accumulators + 128 master sums
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // clear the operand stages once: rows the TMA boxes never write must read as zero in the K reduction
    {
        uint8_t* base_ptr = smem_raw + (smem_base - smem_u32(smem_raw));
        uint4* p4 = reinterpret_cast<uint4*>(base_ptr);
        const uint32_t n16 = ((uint32_t)a.stages + (SPLIT ? 2u : 0u)) * raw_bytes / 16u;
        for (uint32_t i = threadIdx.x; i < n16; i += blockDim.x) p4[i] = make_uint4(0, 0, 0, 0);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy zeros visible to TMA / UMMA
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_dy) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        for (int s = 0; s < a.stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); mbar_init(lo_bar(s), kWgTransformWarps); }
        for (int s = 0; s < 2; ++s) { mbar_init(lo_empty(s), 1); mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(kCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    int tile = blockIdx.x;
    const int nt = tile % a.n_tiles; tile /= a.n_tiles;
    const int mt = tile % a.m_tiles;
    const int tap_tile = tile / a.m_tiles;
    const int tap = a.pair ? 2 * tap_tile : tap_tile;                    // first (or only) tap of this tile
    const bool tap_b = a.pair && (tap + 1 < a.taps);                     // the stacked second tap exists
    const int m0 = mt * 128, k0 = nt * a.n_tile;
    const int split = blockIdx.y;
    const long long c_begin = (long long)split * a.chunks_per_split;
    long long c_end = c_begin + a.chunks_per_split;
    if (c_end > a.chunks_total) c_end = a.chunks_total;
    // which of the 4 dy slots / nsub_b x slots receive TMA data (bit j = slot j)
    uint32_t loaded = 0;
    int b_boxes;
    if (a.blocked) {
        // one box per operand (pair mode: two dy boxes); blocks past the tensor's channel extent arrive as zeros
        loaded = (1u << a.nblk_a) - 1u;
        if (a.pair && tap_b) loaded |= loaded << 2;
        b_boxes = (int)nsub_b;
    } else if (a.pair) {
        const int nb32 = (a.cout + 31) / 32;                             // <= 2
        for (int i = 0; i < nb32; ++i) { loaded |= 1u << i; if (tap_b) loaded |= 1u << (2 + i); }
        b_boxes = (a.cin - k0 + 31) / 32 < (int)nsub_b ? (a.cin - k0 + 31) / 32 : (int)nsub_b;
    } else {
        const int a_boxes = (a.cout - m0 + 31) / 32 < 4 ? (a.cout - m0 + 31) / 32 : 4;
        loaded = (1u << a_boxes) - 1u;
        b_boxes = (a.cin - k0 + 31) / 32 < (int)nsub_b ? (a.cin - k0 + 31) / 32 : (int)nsub_b;
    }
    loaded |= ((1u << b_boxes) - 1u) << 4;
    uint32_t stage_tx = (uint32_t)__popc(loaded) * (uint32_t)a.rows_box * 128u;
    if (PRE) stage_tx = (uint32_t)(a.pre_ablk * ((a.pair && tap_b) ? 2 : 1) + a.pre_bblk) * 2u * (uint32_t)a.rows_box * 128u;
    // (flat: pre_*blk = blocks per box, whole boxes count; timestep boxes: pre_*blk = blocks actually loaded for this tile)
    int pre_na = a.pre_ablk, pre_nb = a.pre_bblk;
    if (PRE && !a.flat) {
        pre_na = ((a.cout - m0 < 128 ? a.cout - m0 : 128) + 63) / 64;
        pre_nb = ((a.cin - k0 < a.n_tile ? a.cin - k0 : a.n_tile) + 63) / 64;
        stage_tx = (uint32_t)(pre_na + pre_nb) * 2u * (uint32_t)a.rows_box * 128u;
    }

    if (warp == 0) {
        {   // warp-uniform loop, elected lane issues the TMA loads (uniform-register operands)
            const bool leader = elect_one_sync() != 0;
            int stage = 0; uint32_t phase = 0;
            for (long long c = c_begin; c < c_end; ++c) {
                const int n = (int)(c / a.chunks_per_sample);
                const int cs = (int)(c - (long long)n * a.chunks_per_sample);
                int a1, a2, b1, b2;
                if (a.flat) { a1 = cs * a.rows_box; a2 = 0; b1 = a1 + (tap - a.pad) * a.v; b2 = 0; }
                else { a1 = 0; a2 = cs * a.tt; b1 = 0; b2 = a.stride * a2 + tap - a.pad; }
                mbar_wait(empty_bar(stage), phase ^ 1u);
                const uint32_t sa = smem_base + (uint32_t)stage * raw_bytes;
                if (leader) {
                    mbar_expect_tx(full_bar(stage), stage_tx);
                    if (PRE && !a.flat) {
                        for (int i = 0; i < pre_na; ++i) {
                            tma_load_5d(sa + (uint32_t)(2 * i) * sub_bytes, &map_dy, full_bar(stage), 0, 0, a2, m0 / 64 + i, n);
                            tma_load_5d(sa + (uint32_t)(2 * i + 1) * sub_bytes, &map_dy_m, full_bar(stage), 0, 0, a2, m0 / 64 + i, n);
                        }
                        for (int j = 0; j < pre_nb; ++j) {
                            tma_load_5d(sa + (uint32_t)(4 + 2 * j) * sub_bytes, &map_x, full_bar(stage), 0, 0, b2, k0 / 64 + j, n);
                            tma_load_5d(sa + (uint32_t)(5 + 2 * j) * sub_bytes, &map_x_m, full_bar(stage), 0, 0, b2, k0 / 64 + j, n);
                        }
                    } else if (PRE) {
                        // dims (64 channels, flat row, piece, 64-channel block, sample); the box covers both pieces and all blocks of the tile
                        tma_load_5d(sa, &map_dy, full_bar(stage), 0, a1, 0, a.pair ? 0 : m0 / 64, n);
                        if (a.pair && tap_b) tma_load_5d(sa + 2u * sub_bytes, &map_dy, full_bar(stage), 0, a1 - a.v, 0, 0, n);
                        tma_load_5d(sa + 4u * sub_bytes, &map_x, full_bar(stage), 0, b1, 0, k0 / 64, n);
                    } else if (a.blocked) {
                        // dims (32 channels, flat row, channel block, sample): the box lands as [block][row][128 B], exactly the slot layout
                        tma_load_4d(sa, &map_dy, full_bar(stage), 0, a1, a.pair ? 0 : m0 / 32, n);
                        if (a.pair && tap_b) tma_load_4d(sa + 2u * sub_bytes, &map_dy, full_bar(stage), 0, a1 - a.v, 0, n);
                        tma_load_4d(sa + 4u * sub_bytes, &map_x, full_bar(stage), 0, b1, k0 / 32, n);
                    } else {
                        if (a.pair) {
                            // slots 0,1: dy rows [a1, ..) for tap 2j; slots 2,3: the same channels V rows earlier for tap 2j+1
                            //   sum_k dy[k - V][co] * x[k + (tap - pad) V][ci] = sum_k' dy[k'][co] * x[k' + (tap + 1 - pad) V][ci]
                            for (int i = 0; i < 4; ++i)
                                if ((loaded >> i) & 1u)
                                    tma_load_4d(sa + i * sub_bytes, &map_dy, full_bar(stage), 32 * (i & 1), i < 2 ? a1 : a1 - a.v, 0, n);
                        } else {
                            for (int i = 0; i < 4; ++i)
                                if ((loaded >> i) & 1u) tma_load_4d(sa + i * sub_bytes, &map_dy, full_bar(stage), m0 + 32 * i, a1, a2, n);
                        }
                        const uint32_t sb = sa + 4u * sub_bytes;
                        for (int j = 0; j < b_boxes; ++j) tma_load_4d(sb + j * sub_bytes, &map_x, full_bar(stage), k0 + 32 * j, b1, b2, n);
                    }
                }
                __syncwarp();
                if (++stage == a.stages) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // all 32 lanes run the warp-uniform control flow and the mbarrier waits, ONE elected lane issues the MMAs / commits, so
        // that ptxas keeps the descriptors in uniform registers (no per-instruction R2UR waterfall; see conv_tc2.cu)
        {
            const bool leader = elect_one_sync() != 0;
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
            // tf32 x tf32 -> f32, A and B MN-major, M = 128, N = n_tile
            constexpr uint32_t kFmt = BF ? 1u : 2u;                        // operand format: BF16 (kind::f16) or TF32
            const uint32_t idesc = (1u << 4) | (kFmt << 7) | (kFmt << 10) | (1u << 15) | (1u << 16) |
                                   ((uint32_t)(a.n_tile >> 3) << 17) | ((128u >> 4) << 24);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            uint32_t d_tmem = tmem_u;
            uint32_t first = 1;
            long long done = 0;
            int sl = 0;
            const long long nchunks = c_end - c_begin;
            const int ksteps = (a.dbg & 2) ? 1 : (BF ? (a.rows_box + 15) / 16 : (a.rows_box + 7) / 8);
            for (long long c = c_begin; c < c_end; ++c) {
                mbar_wait(full_bar(stage), phase);
                if (CONV && !PRE) mbar_wait(lo_bar(stage), phase);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = smem_base + (uint32_t)stage * raw_bytes;
                const uint32_t slo = lo_ring + (uint32_t)sl * raw_bytes;
                const uint64_t da = make_smem_desc_mn(sa, sub_bytes), db = make_smem_desc_mn(sa + 4u * sub_bytes, sub_bytes);
                const uint64_t dalo = make_smem_desc_mn(slo, sub_bytes);
                const uint64_t dblo = make_smem_desc_mn(slo + 4u * sub_bytes, sub_bytes);
                if (leader && BF) {
                    // h pieces in the even slots, m pieces in the odd slots; 64-channel blocks are two slots apart
                    const uint64_t dah = make_smem_desc_mn16(sa, 2u * sub_bytes), dam = make_smem_desc_mn16(sa + sub_bytes, 2u * sub_bytes);
                    const uint64_t dbh = make_smem_desc_mn16(sa + 4u * sub_bytes, 2u * sub_bytes), dbm = make_smem_desc_mn16(sa + 5u * sub_bytes, 2u * sub_bytes);
                    for (int kg = 0; kg < ksteps; ++kg) {
                        const uint64_t ko = (uint64_t)(kg * 128);          // 16 rows = 2048 bytes, in 16-byte units
                        const uint32_t fresh = (kg == 0) ? first : 0u;
                        umma_bf16(d_tmem, dam + ko, dbh + ko, idesc, fresh ^ 1u);
                        umma_bf16(d_tmem, dah + ko, dbm + ko, idesc, 1u);
                        umma_bf16(d_tmem, dah + ko, dbh + ko, idesc, 1u);
                    }
                    umma_commit(empty_bar(stage));
                } else if (leader) {
                    for (int kg = 0; kg < ksteps; ++kg) {
                        const uint64_t ko = (uint64_t)(kg * 64);
                        const uint32_t fresh = (kg == 0) ? first : 0u;
                        if (SPLIT) {
                            umma_tf32(d_tmem, dalo + ko, db + ko, idesc, fresh ^ 1u);
                            umma_tf32(d_tmem, da + ko, dblo + ko, idesc, 1u);
                            umma_tf32(d_tmem, da + ko, db + ko, idesc, 1u);
                        } else {
                            umma_tf32(d_tmem, da + ko, db + ko, idesc, fresh ^ 1u);
                        }
                    }
                    umma_commit(empty_bar(stage));
                    if (SPLIT) umma_commit(lo_empty(sl));
                }
                __syncwarp();
                first = 0;
                if (SPLIT) sl ^= 1;
                if (++stage == a.stages) { stage = 0; phase ^= 1u; }
                ++done;
                if (CONV && (done % a.seg_chunks) == 0 && done < nchunks) {
                    // promote this partial accumulator to the epilogue's fp32 registers, continue in the other TMEM buffer
                    if (leader) umma_commit(tfull_bar(acc));
                    __syncwarp();
                    if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
                    mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    d_tmem = tmem_u + (uint32_t)(acc * 128);
                    first = 1;
                }
            }
            if (leader) umma_commit(tfull_bar(acc));
            __syncwarp();
        }
    } else if (warp < 6) {
        const int q = warp & 3;
        int co, otap;
        if (a.pair) { co = (q & 1) * 32 + lane; otap = tap + (q >> 1); }
        else { co = m0 + q * 32 + lane; otap = tap; }
        const bool store = (co < a.cout) && (otap < a.taps);
        float* out = a.ws + (((long long)split * a.cout + (store ? co : 0)) * a.taps + (store ? otap : 0)) * a.cin + k0;
        const long long nchunks = c_end - c_begin;
        const int nseg = CONV ? (int)((nchunks + a.seg_chunks - 1) / a.seg_chunks) : 1;
        int acc = 0; uint32_t acc_phase = 0;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const uint32_t master = tmem_base + 256u + lane_base;            // SPLIT: fp32 master sums (columns 256..383, n_tile <= 128)
        for (int sg = 0; sg < nseg; ++sg) {
            mbar_wait(tfull_bar(acc), acc_phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t taddr = tmem_base + (uint32_t)(acc * 128) + lane_base;
            const bool last = sg == nseg - 1;
#pragma unroll
            for (int cg = 0; cg < (CONV ? 8 : 16); ++cg) {
                const int c = cg * 16;
                if (c < a.n_tile) {
                    float vals[16];
                    if (CONV) tmem_promote16(taddr + (uint32_t)c, master + (uint32_t)c, sg == 0, !last, vals);
                    else tmem_ld16(taddr + (uint32_t)c, vals);
                    if (last && store) {
#pragma unroll
                        for (int g = 0; g < 4; ++g)
                            if (k0 + c + g * 4 < a.cin)
                                *reinterpret_cast<float4*>(out + c + g * 4) = make_float4(vals[g * 4], vals[g * 4 + 1], vals[g * 4 + 2], vals[g * 4 + 3]);
                    }
                }
            }
            if (CONV && !last) tmem_st_wait();
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
    } else if (BF && !PRE) {
        // BF16x3 converter (kWgTransformWarps warps): slot pair (2j, 2j+1) of 32-channel fp32 blocks -> 64 bf16 channels of h | m in
        // place, one thread per (pair, K row).  Only rows TMA wrote are touched (the pad rows stay zero); a pair whose first slot is
        // never loaded stays zero, a pair with only its first slot loaded gets zero upper channels.
        const int tidx = threadIdx.x - 6 * 32;
        const int npairs = (4 + (int)nsub_b + 1) / 2;
        int stage = 0; uint32_t phase = 0;
        for (long long c = c_begin; c < c_end; ++c) {
            mbar_wait(full_bar(stage), phase);
            const uint32_t sa = smem_base + (uint32_t)stage * raw_bytes;
            for (int idx = tidx; idx < npairs * a.rows_box; idx += kWgTransformWarps * 32) {
                const int pr = idx / a.rows_box, r = idx - pr * a.rows_box;
                if ((loaded >> (2 * pr)) & 1u) {
                    const uint32_t p0 = sa + (uint32_t)(2 * pr) * sub_bytes + (uint32_t)r * 128u;
                    bf16_split_row(p0, p0 + sub_bytes, (uint32_t)(r & 7), ((loaded >> (2 * pr + 1)) & 1u) != 0);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(lo_bar(stage));
            if (++stage == a.stages) { stage = 0; phase ^= 1u; }
        }
    } else if (SPLIT) {
        // operand split (kWgTransformWarps warps): hi = rna_tf32(x) in place, lo = x - hi into the stage's second half.
        // Only the rows TMA wrote are touched (the pad rows stay zero in both halves).
        const int tidx = threadIdx.x - 6 * 32;
        const int nslots = 4 + (int)nsub_b;
        int stage = 0; uint32_t phase = 0;
        int sl = 0; uint32_t pl = 0;
        for (long long c = c_begin; c < c_end; ++c) {
            mbar_wait(full_bar(stage), phase);
            mbar_wait(lo_empty(sl), pl ^ 1u);
            const uint32_t sa = smem_base + (uint32_t)stage * raw_bytes;
            const uint32_t slo = lo_ring + (uint32_t)sl * raw_bytes;
            if (!(a.dbg & 1)) {
                // Slots are `sub_bytes` apart and each holds box_bytes of payload.  When the payload fills the slot (flat layout)
                // the loaded slots of each operand are contiguous, so they are split as two long runs.
                // Slots are `sub_bytes` apart; rows a TMA box does not write are zero in the raw stage and split to (0, 0), so whole
                // slots are processed: the loaded slots of each operand form one contiguous run whenever they are a prefix.
                const uint32_t am = loaded & 15u, na_l = (uint32_t)__popc(am);
                if (am == (1u << na_l) - 1u) {
                    transform_split4(sa, slo, na_l * sub_bytes, tidx, kWgTransformWarps * 32);
                    transform_split4(sa + 4u * sub_bytes, slo + 4u * sub_bytes, (uint32_t)__popc(loaded >> 4) * sub_bytes, tidx, kWgTransformWarps * 32);
                } else {
                    for (int j = 0; j < nslots; ++j)
                        if ((loaded >> j) & 1u)
                            transform_split4(sa + (uint32_t)j * sub_bytes, slo + (uint32_t)j * sub_bytes, sub_bytes, tidx, kWgTransformWarps * 32);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(lo_bar(stage));
            if (++stage == a.stages) { stage = 0; phase ^= 1u; }
            sl ^= 1; if (sl == 0) pl ^= 1u;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kCols) : "memory");
    }
}

struct WgPlan {
    bool ok;
    WgArgs a;
    int splits;
    size_t smem;
};

// split: 0 TF32, 1 3xTF32, 2 BF16x3
static WgPlan plan_wgrad(int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad, int split) {
    WgPlan p;
    p.ok = false;
    if (cin % 4 || cout % 4 || v > 128 || stride > 4) return p;
    WgArgs& a = p.a;
    a.ws = nullptr;
    a.nb = nb; a.t_in = t_in; a.t_out = t_out; a.v = v; a.cin = cin; a.cout = cout; a.taps = taps; a.stride = stride; a.pad = pad;
    a.n_tile = ((cin + 31) / 32) * 32;
    const int n_cap = split ? 128 : 256;          // split: two 128-column TMEM buffers + 128 fp32 promotion registers per thread
    if (a.n_tile > n_cap) a.n_tile = n_cap;
    a.n_tiles = (cin + a.n_tile - 1) / a.n_tile;
    a.m_tiles = (cout + 127) / 128;
    const bool bf = split == 2;
    const int nsub = 4 + (bf ? (a.n_tile / 32 + 1) / 2 * 2 : a.n_tile / 32);     // BF16x3: x slots come in (h, m) pairs
    // Rows per stage.  Every stage costs ~1000-1400 cycles of fixed work (TMA issue, barrier hops, operand split, MMA issue;
    // probes in profiles/r1v, r1w), so stages are as tall as shared memory allows: TF32 four stages of 48 KB; 3xTF32 three raw
    // stages + two lo slots in 200 KB (40 KB each).
    static const int split_kb = probe_env("AGCN_WG_SPLIT_KB") ? atoi(probe_env("AGCN_WG_SPLIT_KB")) : 40;
    a.flat = (stride == 1 && t_in == t_out) ? 1 : 0;
    // strided / shortened outputs load whole timesteps (V rows each): 64 KB stages there, so that two timesteps of a 25-joint
    // skeleton fit one stage instead of one (half the stages, barriers and MMA issue rounds per row)
    int rmax = ((split == 1 ? split_kb : (bf && !a.flat ? 64 : 48)) * 1024) / (nsub * 128);
    rmax = bf ? rmax / 16 * 16 : rmax / 8 * 8;                                     // BF16x3: UMMA K = 16 rows
    if (rmax > 128) rmax = 128;
    if (rmax < 8) return p;
    // two taps per tile when the output channels fill only half of the M = 128 atom (flat layout only: the second tap is
    // the same dy rows V positions earlier)
    a.pair = (a.flat && taps > 1 && cout <= 64) ? 1 : 0;
    a.tap_tiles = a.pair ? (taps + 1) / 2 : taps;
    if (a.flat) {
        a.rows_box = rmax;
        a.rpad = rmax;
        a.tt = 0;
        a.chunks_per_sample = (t_out * v + (a.pair ? v : 0) + a.rows_box - 1) / a.rows_box;
    } else {
        a.tt = rmax / v;
        if (a.tt < 1) { a.tt = 1; }
        while (a.tt * stride > 256) --a.tt;
        a.rows_box = a.tt * v;
        a.rpad = bf ? (a.rows_box + 15) / 16 * 16 : (a.rows_box + 7) / 8 * 8;
        if ((size_t)nsub * a.rpad * 128 * (split == 1 ? 2 : 1) > 96 * 1024) return p;
        a.chunks_per_sample = (t_out + a.tt - 1) / a.tt;
    }
    a.chunks_total = (long long)nb * a.chunks_per_sample;
    a.seg_chunks = (bf ? 512 : 256) / a.rows_box;      // rows per accumulator segment: <= 32 K steps x 3 chained MMAs
    if (a.seg_chunks < 1) a.seg_chunks = 1;
    const size_t raw_stage = (size_t)nsub * a.rpad * 128;
    int stages = (int)((200 * 1024 - (split == 1 ? 2 * raw_stage : 0)) / raw_stage);     // 3xTF32: two extra slots hold the lo residuals
    if (stages > kWgStages) stages = kWgStages;
    if (stages < 2) return p;
    a.stages = stages;
    // one resident wave: (tiles x splits) CTAs <= 148 SMs (1 CTA / SM), every CTA streams an equal share of the row chunks
    const long long tiles = (long long)a.tap_tiles * a.m_tiles * a.n_tiles;
    long long splits = kNumSMs / tiles;
    if (splits > a.chunks_total) splits = a.chunks_total;
    if (splits < 1) splits = 1;
    a.chunks_per_split = (a.chunks_total + splits - 1) / splits;
    splits = (a.chunks_total + a.chunks_per_split - 1) / a.chunks_per_split;
    p.splits = (int)splits;
    p.smem = (size_t)(stages + (split == 1 ? 2 : 0)) * raw_stage + 1024 + kWgBarBytes;
    p.ok = true;
    return p;
}

}  // namespace tc
}  // namespace agcn

using namespace agcn;

// ---- weight gradient on tensor cores; returns AGCN_ERR_UNSUPPORTED for shapes outside the path
size_t agcn_conv_wgrad_tc_workspace_floats(int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad, int split) {
    agcn::tc::WgPlan p = agcn::tc::plan_wgrad(nb, t_in, t_out, v, cin, cout, taps, stride, pad, split);
    if (!p.ok) return 0;
    return (size_t)p.splits * cout * taps * cin;
}

int agcn_conv_wgrad_tc(const float* dy, const float* x, float* ws, int* splits_out,
                       int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad, int split, void* stream) {
    using namespace agcn::tc;
    if (!aligned16(dy) || !aligned16(x) || !aligned16(ws)) return AGCN_ERR_UNSUPPORTED;
    WgPlan p = plan_wgrad(nb, t_in, t_out, v, cin, cout, taps, stride, pad, split);
    if (!p.ok) return AGCN_ERR_UNSUPPORTED;
    EncodeTiledFn enc = encode_fn();
    if (!enc) return fail(AGCN_ERR_CUDA, "agcn_conv_wgrad_tc: cuTensorMapEncodeTiled is not available from the driver");
    WgArgs& a = p.a;
    a.ws = ws;
    static const int dbg = probe_env("AGCN_WG_DEBUG") ? atoi(probe_env("AGCN_WG_DEBUG")) : 0;
    a.dbg = dbg;
    CUtensorMap map_dy, map_x;
    static const bool no_blocked = probe_env("AGCN_WG_NOBLOCK") != nullptr;
    a.blocked = (!no_blocked && a.flat && cin % 32 == 0 && cout % 32 == 0) ? 1 : 0;
    a.nblk_a = a.pair ? cout / 32 : ((cout + 31) / 32 < 4 ? (cout + 31) / 32 : 4);
    auto encode = [&](CUtensorMap* m, const float* ptr, int c, int t, int box1, int box2, int es2) -> CUresult {
        cuuint64_t dims[4]; cuuint64_t strides[3]; cuuint32_t box[4]; cuuint32_t estr[4] = {1, 1, 1, 1};
        if (a.blocked) {
            // (32 channels, flat row, channel block, sample): the channel block is a dimension of its own (stride 128 B, smaller
            // than the row stride), so ONE box covers all 32-channel blocks of the tile -- the per-box issue cost of the TMA
            // producer thread (~180 cycles, profiles/r1v) was the floor of this kernel
            dims[0] = 32; dims[1] = (cuuint64_t)t * v; dims[2] = (cuuint64_t)c / 32; dims[3] = nb;
            strides[0] = (cuuint64_t)c * 4; strides[1] = 128; strides[2] = (cuuint64_t)t * v * c * 4;
            box[0] = 32; box[1] = box1; box[2] = (cuuint32_t)box2; box[3] = 1;
        } else if (a.flat) {
            dims[0] = c; dims[1] = (cuuint64_t)t * v; dims[2] = 1; dims[3] = nb;
            strides[0] = (cuuint64_t)c * 4; strides[1] = (cuuint64_t)t * v * c * 4; strides[2] = (cuuint64_t)t * v * c * 4;
            box[0] = 32; box[1] = box1; box[2] = 1; box[3] = 1;
        } else {
            dims[0] = c; dims[1] = v; dims[2] = t; dims[3] = nb;
            strides[0] = (cuuint64_t)c * 4; strides[1] = (cuuint64_t)v * c * 4; strides[2] = (cuuint64_t)t * v * c * 4;
            box[0] = 32; box[1] = v; box[2] = box2; box[3] = 1;
            estr[2] = es2;
        }
        // TF32 operands are read by the MMA as they land (32-byte-atom swizzle, the only MN-major tf32 layout); the BF16x3
        // converter reads plain 128B-swizzled rows
        return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, split == 2 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    };
    CUresult r = encode(&map_dy, dy, cout, t_out, a.rows_box, a.blocked ? a.nblk_a : a.tt, 1);
    if (r == CUDA_SUCCESS) r = encode(&map_x, x, cin, t_in, a.rows_box, a.blocked ? a.n_tile / 32 : a.tt * stride, stride);
    if (r != CUDA_SUCCESS && a.blocked) {          // driver refused the blocked maps: fall back to one box per 32-channel block
        a.blocked = 0;
        r = encode(&map_dy, dy, cout, t_out, a.rows_box, a.tt, 1);
        if (r == CUDA_SUCCESS) r = encode(&map_x, x, cin, t_in, a.rows_box, a.tt * stride, stride);
    }
    if (r != CUDA_SUCCESS) return fail(AGCN_ERR_CUDA, "agcn_conv_wgrad_tc: cuTensorMapEncodeTiled failed with %d", (int)r);
    {   // per call: the attribute is per device / context, a process-wide flag would skip the second GPU
        cudaError_t e = cudaFuncSetAttribute(wgrad_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);
        if (e != cudaSuccess) return fail(AGCN_ERR_CUDA, "agcn_conv_wgrad_tc: %s", cudaGetErrorString(e));
    }
    dim3 grid((unsigned)(a.tap_tiles * a.m_tiles * a.n_tiles), (unsigned)p.splits);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (split == 2) wgrad_tc_kernel<2><<<grid, kWgThreadsSplit, p.smem, st>>>(map_dy, map_x, map_dy, map_x, a);
    else if (split) wgrad_tc_kernel<1><<<grid, kWgThreadsSplit, p.smem, st>>>(map_dy, map_x, map_dy, map_x, a);
    else wgrad_tc_kernel<0><<<grid, kThreads, p.smem, st>>>(map_dy, map_x, map_dy, map_x, a);
    *splits_out = p.splits;
    return check_launch("agcn_conv_wgrad_tc");
}

// ---- the same on operands that arrive split: dy_split = [2][nb * t_out * v][cout], x_split = [2][nb * t_in * v][cin] bf16 (plane 0 = h =
// bf16(x), plane 1 = m = bf16(x - h)).  Channel counts multiples of 64.  AGCN_ERR_UNSUPPORTED otherwise.
int agcn_conv_wgrad_tc_presplit(const uint16_t* dy_split, const uint16_t* x_split, float* ws, int* splits_out,
                                int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad, void* stream) {
    using namespace agcn::tc;
    if (cin % 64 || cout % 64 || !aligned16(dy_split) || !aligned16(x_split) || !aligned16(ws)) return AGCN_ERR_UNSUPPORTED;
    WgPlan p = plan_wgrad(nb, t_in, t_out, v, cin, cout, taps, stride, pad, 2);
    if (!p.ok || p.a.n_tile % 64) return AGCN_ERR_UNSUPPORTED;
    EncodeTiledFn enc = encode_fn();
    if (!enc) return fail(AGCN_ERR_CUDA, "agcn_conv_wgrad_tc_presplit: cuTensorMapEncodeTiled is not available from the driver");
    WgArgs& a = p.a;
    a.ws = ws; a.dbg = 0; a.blocked = 0; a.nblk_a = 0;
    a.pre_ablk = a.pair ? 1 : (cout < 128 ? 1 : 2);
    a.pre_bblk = a.n_tile / 64;
    CUtensorMap map_dy, map_x, map_dy_m, map_x_m;
    CUresult r;
    if (a.flat) {
        auto encode = [&](CUtensorMap* m, const uint16_t* ptr, int c, int nblk) -> CUresult {
            // dims (64 channels, flat row of the sample, piece, 64-channel block, sample)
            const cuuint64_t rows = (cuuint64_t)t_out * v, plane = (cuuint64_t)nb * rows * c * 2;
            cuuint64_t dims[5] = {64, rows, 2, (cuuint64_t)c / 64, (cuuint64_t)nb};
            cuuint64_t strides[4] = {(cuuint64_t)c * 2, plane, 128, rows * c * 2};
            cuuint32_t box[5] = {64, (cuuint32_t)a.rows_box, 2, (cuuint32_t)nblk, 1};
            cuuint32_t estr[5] = {1, 1, 1, 1, 1};
            return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<uint16_t*>(ptr), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        };
        r = encode(&map_dy, dy_split, cout, a.pre_ablk);
        if (r == CUDA_SUCCESS) r = encode(&map_x, x_split, cin, a.pre_bblk);
        map_dy_m = map_dy; map_x_m = map_x;
    } else {
        auto encode = [&](CUtensorMap* m, const uint16_t* ptr, int c, int t, int box_t, int es_t) -> CUresult {
            // one piece: dims (64 channels, v, t, 64-channel block, sample); whole timesteps per box, element stride on t for the input
            cuuint64_t dims[5] = {64, (cuuint64_t)v, (cuuint64_t)t, (cuuint64_t)c / 64, (cuuint64_t)nb};
            cuuint64_t strides[4] = {(cuuint64_t)c * 2, (cuuint64_t)v * c * 2, 128, (cuuint64_t)t * v * c * 2};
            cuuint32_t box[5] = {64, (cuuint32_t)v, (cuuint32_t)box_t, 1, 1};
            cuuint32_t estr[5] = {1, 1, (cuuint32_t)es_t, 1, 1};
            return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<uint16_t*>(ptr), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        };
        const size_t plane_dy = (size_t)nb * t_out * v * cout, plane_x = (size_t)nb * t_in * v * cin;
        r = encode(&map_dy, dy_split, cout, t_out, a.tt, 1);
        if (r == CUDA_SUCCESS) r = encode(&map_dy_m, dy_split + plane_dy, cout, t_out, a.tt, 1);
        if (r == CUDA_SUCCESS) r = encode(&map_x, x_split, cin, t_in, a.tt * stride, stride);
        if (r == CUDA_SUCCESS) r = encode(&map_x_m, x_split + plane_x, cin, t_in, a.tt * stride, stride);
    }
    if (r != CUDA_SUCCESS) return fail(AGCN_ERR_CUDA, "agcn_conv_wgrad_tc_presplit: cuTensorMapEncodeTiled failed with %d", (int)r);
    cudaError_t e = cudaFuncSetAttribute(wgrad_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);
    if (e != cudaSuccess) return fail(AGCN_ERR_CUDA, "agcn_conv_wgrad_tc_presplit: %s", cudaGetErrorString(e));
    dim3 grid((unsigned)(a.tap_tiles * a.m_tiles * a.n_tiles), (unsigned)p.splits);
    wgrad_tc_kernel<3><<<grid, kThreads, p.smem, static_cast<cudaStream_t>(stream)>>>(map_dy, map_x, map_dy_m, map_x_m, a);
    *splits_out = p.splits;
    return check_launch("agcn_conv_wgrad_tc_presplit");
}
