// cv_attn_bwd: backward of the fused dense attention (autograd of standard_attention,
// /root/reference/mpu/sparse_transformer.py:652-673, which the reference gets from torch autograd over
// materialised [b, np, s, s] tensors).  Recomputes P from Q, K and the saved log-sum-exp; nothing of
// size [s, s] reaches HBM.
//
//   P = exp(S - lse),  S = scale * Q K^T (masked entries: -10000, gradient 0)
//   dV = P^T dO        dP = dO V^T        dS = P o (dP - D),  D = rowsum(dO o O)
//   dQ = scale * dS K  dK = scale * dS^T Q
//
// One CTA per (128-key block, head, batch) loops over the query blocks that can see it.  All five products
// run on tcgen05 with TMEM accumulators; every operand is used in place from 128B-swizzled TMA tiles, in
// K-major or MN-major form as the product needs (the same Q / dO / K tiles serve both):
//   S^T  = K Q^T      (A = K   K-major, B = Q  K-major)   [keys x queries]
//   dP^T = V dO^T     (A = V   K-major, B = dO K-major)
//   dV  += P^T dO     (A = P^T K-major (smem, written by the softmax warps), B = dO MN-major)
//   dK  += dS^T Q     (A = dS^T K-major (smem),                               B = Q  MN-major)
//   dQ_i = dS K       (A = dS^T read MN-major,                                B = K  MN-major)
// dV / dK stay in TMEM for the whole loop; dQ tiles are reduced into an fp32 buffer with vector red.add.
#include "common.cuh"
#include "host.h"
#include "../../include/cogview_b200.h"

namespace {
using namespace cv;

constexpr int BLK = 128;
constexpr int HD = 64;
constexpr int TILE_BYTES = BLK * HD * 2;      // 16 KB: one [128 x 64] bf16 tile
constexpr int PT_BYTES = BLK * BLK * 2;       // 32 KB: [128 keys x 128 queries] bf16
constexpr int QDO_STAGES = 2;
constexpr int SMEM_BYTES = 2 * TILE_BYTES /*K,V*/ + QDO_STAGES * 2 * TILE_BYTES /*Q,dO*/ + 2 * PT_BYTES /*P^T,dS^T*/ +
                           QDO_STAGES * 3 * BLK * 4 /*lse2, D, band start*/ + 1024 + 256;
enum { MODE_DENSE = 0, MODE_BAND = 1, MODE_PIVOT = 2 };
constexpr int NUM_THREADS = 320;     // TMA warp, MMA warp, 8 compute warps (two threads per key row)
constexpr float LOG2E = 1.4426950408889634f;

struct BwdParams {
    int b, heads, s;
    int sep_eff;
    float scale, scale_log2;
    const float* lse;    // [b, heads, s]
    const float* delta;  // [b, heads, s]
    float* dq_acc;       // [b, s, heads*HD] fp32, zero-initialised
    __nv_bfloat16* dqkv; // [b, s, 3*heads*HD]
    const uint32_t* drop_mask;  // keep bits written by the forward, key-major ([b, heads, keep_rows, nqb, 4]: the 128 query
                                // bits of (key, query block) are one 16-byte load for the thread that owns the key) or null
    int keep_rows;              // key rows per (batch, head) of drop_mask: nqb*128 (dense, band pass), npt*128 (pivot pass)
    float drop_scale;           // 1 / (1 - p)
    // sparse training attention (mpu/sparse_transformer.py:675-725), two launches that share lse / delta / dq_acc:
    //   MODE_BAND : keys = the sequence, key j visible to query i iff band_start(i) <= j <= i
    //   MODE_PIVOT: keys = the gathered pivots (sk = n_piv rows), pivot visible iff piv_pos < band_start(i),
    //               scores carry + log(s / n_piv); dK / dV rows go to the gathered scratch (kv_rows = n_piv)
    int sk, kv_rows, sp_w, sp_times;
    const int* piv_pos;         // [b, sk]
    float piv_bias_log2;
};

__device__ __forceinline__ int band_start(int i, int w, int times) {
    const int g = i / w - times + 1;
    return g > 0 ? g * w : 0;
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
                 : "memory");
}

template <int MODE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO, const BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sK = smem;
    uint8_t* sV = sK + TILE_BYTES;
    uint8_t* sQDO = sV + TILE_BYTES;                               // stage s: Q then dO
    uint8_t* sPT = sQDO + QDO_STAGES * 2 * TILE_BYTES;
    uint8_t* sDST = sPT + PT_BYTES;
    float* sLse = reinterpret_cast<float*>(sDST + PT_BYTES);       // [stages][128]
    float* sDelta = sLse + QDO_STAGES * BLK;
    int* sBand = reinterpret_cast<int*>(sDelta + QDO_STAGES * BLK);   // [stages][128] band_start of the tile's queries
    uint64_t* bars = reinterpret_cast<uint64_t*>(sBand + QDO_STAGES * BLK);
    uint64_t* kv_full = bars;                  // 1
    uint64_t* qdo_full = bars + 1;             // [2]
    uint64_t* qdo_empty = qdo_full + QDO_STAGES;
    uint64_t* sdp_full = qdo_empty + QDO_STAGES;   // 1: S^T and dP^T ready in TMEM
    uint64_t* pds_full = sdp_full + 1;             // 1: P^T / dS^T written to smem (and S^T/dP^T TMEM consumed)
    uint64_t* pds_free = pds_full + 1;             // 1: MMAs reading P^T / dS^T smem retired
    uint64_t* dq_full = pds_free + 1;              // 1
    uint64_t* dq_free = dq_full + 1;               // 1
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(dq_free + 1);

    const int warp_idx = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kb = blockIdx.x, head = blockIdx.y, batch = blockIdx.z;
    const int k0 = kb * BLK;
    const int nqb = (p.s + BLK - 1) / BLK;
    // query blocks that can see a key of this block
    int i_start = (k0 < p.sep_eff) ? 0 : kb, i_end = nqb - 1;
    if (MODE == MODE_BAND) {          // queries i with band_start(i) <= j <= i
        i_start = kb;
        i_end = min(nqb - 1, (((k0 + BLK - 1) / p.sp_w + p.sp_times) * p.sp_w - 1) / BLK);
    } else if (MODE == MODE_PIVOT) {  // band_start(i) > 0  <=>  i >= sp_times * sp_w   (the host checks this is < s)
        i_start = (p.sp_times * p.sp_w) / BLK;
    }
    const int ntiles = i_end - i_start + 1;

    if (warp_idx == 0 && lane == 0) {
        tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmDO);
        mbar_init(kv_full, 1);
        for (int i = 0; i < QDO_STAGES; ++i) { mbar_init(&qdo_full[i], 1); mbar_init(&qdo_empty[i], 1); }
        mbar_init(sdp_full, 1);
        mbar_init(pds_full, 256);
        mbar_init(pds_free, 1);
        mbar_init(dq_full, 1);
        mbar_init(dq_free, 256);
        fence_barrier_init();
    }
    if (warp_idx == 1) tmem_alloc<512>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    constexpr uint32_t TM_ST = 0, TM_DPT = 128, TM_DV = 256, TM_DK = 320, TM_DQ = 384;

    if (warp_idx == 0) {
        if (lane == 0) {
            mbar_expect_tx(kv_full, 2 * TILE_BYTES);
            tma_load_3d(sK, &tmK, kv_full, head * HD, k0, batch);
            tma_load_3d(sV, &tmV, kv_full, head * HD, k0, batch);
            int stage = 0; uint32_t phase = 0;
            for (int t = 0; t < ntiles; ++t) {
                const int q0 = (i_start + t) * BLK;
                mbar_wait(&qdo_empty[stage], phase ^ 1);
                uint8_t* sQ = sQDO + stage * 2 * TILE_BYTES;
                mbar_expect_tx(&qdo_full[stage], 2 * TILE_BYTES);
                tma_load_3d(sQ, &tmQ, &qdo_full[stage], head * HD, q0, batch);
                tma_load_3d(sQ + TILE_BYTES, &tmDO, &qdo_full[stage], head * HD, q0, batch);
                if (++stage == QDO_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp_idx == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc_s = make_idesc_bf16(BLK, BLK, 0, 0);
            constexpr uint32_t idesc_acc = make_idesc_bf16(BLK, HD, 0, 1);   // A K-major (smem P^T/dS^T), B MN-major
            constexpr uint32_t idesc_dq = make_idesc_bf16(BLK, HD, 1, 1);    // A MN-major (dS^T read as dS), B MN-major
            const uint32_t k_addr = smem_u32(sK), v_addr = smem_u32(sV);
            const uint32_t pt_addr = smem_u32(sPT), dst_addr = smem_u32(sDST);
            auto issue_sdp = [&](int stage) {
                const uint32_t q_addr = smem_u32(sQDO + stage * 2 * TILE_BYTES);
                const uint32_t do_addr = q_addr + TILE_BYTES;
#pragma unroll
                for (int k = 0; k < HD / 16; ++k)
                    umma_f16(tmem_base + TM_ST, make_smem_desc_sw128(k_addr + k * 32, 0, 1024),
                             make_smem_desc_sw128(q_addr + k * 32, 0, 1024), idesc_s, k != 0);
#pragma unroll
                for (int k = 0; k < HD / 16; ++k)
                    umma_f16(tmem_base + TM_DPT, make_smem_desc_sw128(v_addr + k * 32, 0, 1024),
                             make_smem_desc_sw128(do_addr + k * 32, 0, 1024), idesc_s, k != 0);
                umma_commit(sdp_full);
            };
            mbar_wait(kv_full, 0);
            int stage = 0; uint32_t phase = 0;
            mbar_wait(&qdo_full[0], 0);
            tc_fence_after();
            issue_sdp(0);
            for (int t = 0; t < ntiles; ++t) {
                mbar_wait(pds_full, t & 1);           // P^T / dS^T in smem; S^T / dP^T TMEM consumed
                if (t > 0) mbar_wait(dq_free, (t - 1) & 1);   // previous dQ tile drained from TMEM
                tc_fence_after();
                const uint32_t q_addr = smem_u32(sQDO + stage * 2 * TILE_BYTES);
                const uint32_t do_addr = q_addr + TILE_BYTES;
                // dQ first: the softmax warps are waiting for it, and its read-out (TMEM -> red.add) then overlaps dV / dK
#pragma unroll
                for (int k = 0; k < BLK / 16; ++k)     // reduction over the 128 keys of this block
                    umma_f16(tmem_base + TM_DQ, make_smem_desc_sw128(dst_addr + k * 2048, BLK * 128, 1024),
                             make_smem_desc_sw128(k_addr + k * 2048, BLK * 128, 1024), idesc_dq, k != 0);
                umma_commit(dq_full);
#pragma unroll
                for (int k = 0; k < BLK / 16; ++k) {   // reduction over the 128 queries of this tile
                    const uint32_t a_off = (k >> 2) * (BLK * 128) + (k & 3) * 32;
                    umma_f16(tmem_base + TM_DV, make_smem_desc_sw128(pt_addr + a_off, 0, 1024),
                             make_smem_desc_sw128(do_addr + k * 2048, BLK * 128, 1024), idesc_acc, (t | k) != 0);
                    umma_f16(tmem_base + TM_DK, make_smem_desc_sw128(dst_addr + a_off, 0, 1024),
                             make_smem_desc_sw128(q_addr + k * 2048, BLK * 128, 1024), idesc_acc, (t | k) != 0);
                }
                umma_commit(&qdo_empty[stage]);
                umma_commit(pds_free);
                if (++stage == QDO_STAGES) { stage = 0; phase ^= 1; }
                if (t + 1 < ntiles) {
                    mbar_wait(&qdo_full[stage], phase);
                    tc_fence_after();
                    issue_sdp(stage);
                }
            }
        }
    } else {
        // 8 warps: warp w works on TMEM lane quadrant w % 4 (key rows 32 (w % 4) .. +31, one per lane); warps 2-5 take
        // query columns 0-63 of every tile (and dQ / dK), warps 6-9 columns 64-127 (and dV): the per-tile chain of a
        // thread is halved and every scheduler has two of these warps to overlap.  No exchange is needed between the two
        // threads of a row — lse, delta and the band starts come from shared memory.
        const int q = warp_idx & 3;
        const int hf = (warp_idx - 2) >> 2;
        const int row = q * 32 + lane;             // key row within the block
        const int kj = k0 + row;
        const int epi_tid = threadIdx.x - 64;      // 0..255; the first 128 stage the per-query statistics
        const uint32_t lane_addr = tmem_base + (uint32_t(q * 32) << 16);
        const float masked_val = -10000.0f * LOG2E;
        const int my_pos = (MODE == MODE_PIVOT) ? (kj < p.sk ? p.piv_pos[(size_t)batch * p.sk + kj] : 0x7fffffff) : 0;
        const size_t stat_base = ((size_t)batch * p.heads + head) * p.s;
        const size_t keep_base = ((size_t)batch * p.heads + head) * (size_t)p.keep_rows;   // key rows padded to blocks
        int stage = 0;
        float pre_lse, pre_delta;
        uint4 pre_keep = make_uint4(0, 0, 0, 0);
        {
            const int qn = i_start * BLK + (epi_tid & (BLK - 1));
            pre_lse = (qn < p.s) ? p.lse[stat_base + qn] * LOG2E : 0.f;
            pre_delta = (qn < p.s) ? p.delta[stat_base + qn] : 0.f;
            if (p.drop_mask != nullptr)
                pre_keep = *reinterpret_cast<const uint4*>(p.drop_mask + ((keep_base + kj) * (size_t)nqb + i_start) * 4);
        }
        for (int t = 0; t < ntiles; ++t) {
            const int q0 = (i_start + t) * BLK;
            // lse (log2 domain), delta and keep bits of this query block were fetched one tile ahead (registers):
            // publish them, then start the fetch for the next tile so its global-load latency is off the critical path
            if (hf == 0) {
                sLse[stage * BLK + epi_tid] = pre_lse;
                sDelta[stage * BLK + epi_tid] = pre_delta;
                if (MODE != MODE_DENSE) sBand[stage * BLK + epi_tid] = band_start(q0 + epi_tid, p.sp_w, p.sp_times);
            }
            const uint4 kw = pre_keep;                  // this key's keep bits over the 128 queries of the tile
            if (t + 1 < ntiles) {
                const int qn = q0 + BLK + (epi_tid & (BLK - 1));
                pre_lse = (qn < p.s) ? p.lse[stat_base + qn] * LOG2E : 0.f;
                pre_delta = (qn < p.s) ? p.delta[stat_base + qn] : 0.f;
                if (p.drop_mask != nullptr)
                    pre_keep = *reinterpret_cast<const uint4*>(p.drop_mask +
                                                               ((keep_base + kj) * (size_t)nqb + i_start + t + 1) * 4);
            }
            named_bar_sync(1, 256);
            mbar_wait(sdp_full, t & 1);
            tc_fence_after();
            if (t > 0) mbar_wait(pds_free, (t - 1) & 1);   // MMAs of the previous tile no longer read P^T / dS^T
            bool full_vis = (q0 + BLK <= p.s) && (k0 + BLK <= p.s) &&
                            ((k0 + BLK <= p.sep_eff) || (k0 + BLK - 1 <= q0));
            if (MODE == MODE_BAND)      // every key of the block inside the band of every query of the tile
                full_vis = (q0 + BLK <= p.s) && (k0 + BLK - 1 <= q0) &&
                           (k0 >= band_start(q0 + BLK - 1, p.sp_w, p.sp_times));
            if (MODE == MODE_PIVOT) full_vis = false;
            const int* bnd = sBand + stage * BLK;
            const float* lse2 = sLse + stage * BLK;
            const float* dlt = sDelta + stage * BLK;
            const bool use_drop = p.drop_mask != nullptr;
            uint8_t* prow = sPT + row * 128;
            uint8_t* drow = sDST + row * 128;
#pragma unroll 2
            for (int c = hf * 2; c < hf * 2 + 2; ++c) {      // this thread's 64 query columns
                uint32_t sr[32], dr[32];
                tmem_ld_x32(lane_addr + TM_ST + c * 32, sr);
                tmem_ld_x32(lane_addr + TM_DPT + c * 32, dr);
                tmem_ld_wait();
                float pv[32], dv[32];
                const uint32_t kwc = c == 0 ? kw.x : (c == 1 ? kw.y : (c == 2 ? kw.z : kw.w));
                if (full_vis && use_drop) {            // interior tile with dropout: branch-free, bit i of kwc = query col
                    const float ds = p.drop_scale;
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const int col = c * 32 + i;
                        const bool keep = (kwc >> i) & 1u;
                        const float pr = exp2f(__uint_as_float(sr[i]) * p.scale_log2 - lse2[col]);
                        // dP flows back through the keep mask; dV sees the dropped probabilities
                        const float dp = keep ? __uint_as_float(dr[i]) * ds : 0.f;
                        pv[i] = keep ? pr * ds : 0.f;
                        dv[i] = pr * (dp - dlt[col]) * p.scale;
                    }
                } else if (full_vis) {                 // interior tile, no dropout: branch-free inner loop
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const int col = c * 32 + i;
                        const float pr = exp2f(__uint_as_float(sr[i]) * p.scale_log2 - lse2[col]);
                        pv[i] = pr;
                        dv[i] = pr * (__uint_as_float(dr[i]) - dlt[col]) * p.scale;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const int col = c * 32 + i;
                        const int qi = q0 + col;
                        float s2 = __uint_as_float(sr[i]) * p.scale_log2;
                        float pr;
                        if (full_vis) {
                            pr = exp2f(s2 - lse2[col]);
                        } else if (MODE == MODE_PIVOT) {
                            const bool vis = my_pos < bnd[col];
                            s2 = vis ? s2 + p.piv_bias_log2 : masked_val;
                            pr = (kj < p.sk && qi < p.s) ? exp2f(s2 - lse2[col]) : 0.f;
                        } else {
                            const bool vis = (MODE == MODE_BAND) ? (kj >= bnd[col] && kj <= qi)
                                                                 : ((kj < p.sep_eff) || (kj <= qi));
                            if (!vis) s2 = masked_val;
                            pr = (kj < p.s && qi < p.s) ? exp2f(s2 - lse2[col]) : 0.f;
                        }
                        float dp = __uint_as_float(dr[i]);
                        float pdrop = pr;
                        if (use_drop) {   // dP flows back through the keep mask; dV sees the dropped probabilities
                            const bool keep = (kwc >> i) & 1u;
                            dp = keep ? dp * p.drop_scale : 0.f;
                            pdrop = keep ? pr * p.drop_scale : 0.f;
                        }
                        pv[i] = pdrop;
                        dv[i] = pr * (dp - dlt[col]) * p.scale;
                    }
                }
#pragma unroll
                for (int g = 0; g < 4; ++g) {          // 4 chunks of 8 queries (16 bytes)
                    uint4 a, d;
                    a.x = pack_bf16x2(pv[g * 8 + 0], pv[g * 8 + 1]); a.y = pack_bf16x2(pv[g * 8 + 2], pv[g * 8 + 3]);
                    a.z = pack_bf16x2(pv[g * 8 + 4], pv[g * 8 + 5]); a.w = pack_bf16x2(pv[g * 8 + 6], pv[g * 8 + 7]);
                    d.x = pack_bf16x2(dv[g * 8 + 0], dv[g * 8 + 1]); d.y = pack_bf16x2(dv[g * 8 + 2], dv[g * 8 + 3]);
                    d.z = pack_bf16x2(dv[g * 8 + 4], dv[g * 8 + 5]); d.w = pack_bf16x2(dv[g * 8 + 6], dv[g * 8 + 7]);
                    const int chunk = c * 4 + g;           // 16-byte chunk index along the 128 queries
                    const int sub = chunk >> 3, cc = chunk & 7;
                    const int off = sub * (BLK * 128) + ((cc ^ (row & 7)) << 4);
                    *reinterpret_cast<uint4*>(prow + off) = a;
                    *reinterpret_cast<uint4*>(drow + off) = d;
                }
            }
            fence_proxy_async_smem();
            tc_fence_before();
            mbar_arrive(pds_full);
            // dQ tile of this (query block, key block) pair
            mbar_wait(dq_full, t & 1);
            tc_fence_after();
            {
                uint32_t r[HD / 2];                    // this thread's 32 of the row's 64 dims
                tmem_ld_x32(lane_addr + TM_DQ + hf * (HD / 2), r);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(dq_free);
                const int qi = q0 + row;               // here `row` indexes the query (dQ tile rows are queries)
                if (qi < p.s) {
                    float* dst = p.dq_acc + ((size_t)batch * p.s + qi) * (p.heads * HD) + head * HD + hf * (HD / 2);
#pragma unroll
                    for (int i = 0; i < HD / 2; i += 4)
                        red_add_v4(dst + i, __uint_as_float(r[i]), __uint_as_float(r[i + 1]),
                                   __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
                }
            }
            if (++stage == QDO_STAGES) stage = 0;
        }
        // dK / dV of this key block: complete once the last tile's dV / dK MMAs retired (its pds_free commit)
        mbar_wait(pds_free, (ntiles - 1) & 1);
        tc_fence_after();
        // (tcgen05.ld is warp-collective: every lane loads, only in-range rows store)
        {
            const int H3 = 3 * p.heads * HD;
            const bool row_ok = kj < p.kv_rows;
            __nv_bfloat16* base = p.dqkv + ((size_t)batch * p.kv_rows + (row_ok ? kj : 0)) * H3 + head * HD;
            {
                const int which = hf;                  // warps 2-5 store dK, warps 6-9 dV
                uint32_t r[HD];
                uint32_t (&r0)[32] = *reinterpret_cast<uint32_t(*)[32]>(&r[0]);
                uint32_t (&r1)[32] = *reinterpret_cast<uint32_t(*)[32]>(&r[32]);
                const uint32_t col = which == 0 ? TM_DK : TM_DV;
                tmem_ld_x32(lane_addr + col, r0);
                tmem_ld_x32(lane_addr + col + 32, r1);
                tmem_ld_wait();
                __nv_bfloat16* dst = base + (which == 0 ? 1 : 2) * (p.heads * HD);
                if (row_ok) {
#pragma unroll
                for (int c = 0; c < HD / 8; ++c) {
                    uint4 pk;
                    pk.x = pack_bf16x2(__uint_as_float(r[c * 8 + 0]), __uint_as_float(r[c * 8 + 1]));
                    pk.y = pack_bf16x2(__uint_as_float(r[c * 8 + 2]), __uint_as_float(r[c * 8 + 3]));
                    pk.z = pack_bf16x2(__uint_as_float(r[c * 8 + 4]), __uint_as_float(r[c * 8 + 5]));
                    pk.w = pack_bf16x2(__uint_as_float(r[c * 8 + 6]), __uint_as_float(r[c * 8 + 7]));
                    *reinterpret_cast<uint4*>(dst + c * 8) = pk;
                }
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp_idx == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

// delta[b, head, q] = sum_d dO[b, q, head, d] * O[b, q, head, d]
__global__ void attn_bwd_delta_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o,
                                      float* __restrict__ delta, int b, int heads, int s) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (batch, q, head), head fastest
    if (idx >= b * s * heads) return;
    const int head = idx % heads;
    const int tok = idx / heads;
    const uint4* po = reinterpret_cast<const uint4*>(o + (size_t)tok * heads * HD + head * HD);
    const uint4* pd = reinterpret_cast<const uint4*>(d_o + (size_t)tok * heads * HD + head * HD);
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < HD / 8; ++i) {
        uint4 a = po[i], c = pd[i];
        const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
        const __nv_bfloat162* pc = reinterpret_cast<const __nv_bfloat162*>(&c);
#pragma unroll
        for (int t = 0; t < 4; ++t)
            acc += __low2float(pa[t]) * __low2float(pc[t]) + __high2float(pa[t]) * __high2float(pc[t]);
    }
    const int bi = tok / s, qi = tok % s;
    delta[((size_t)bi * heads + head) * s + qi] = acc;
}

// dqkv[:, 0:h] = bf16(dq_acc)
__global__ void attn_bwd_dq_store_kernel(const float* __restrict__ dq, __nv_bfloat16* __restrict__ dqkv, size_t rows,
                                         int h) {
    const size_t n4 = rows * (size_t)(h / 4);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / (h / 4);
        const int c = (int)(i % (h / 4)) * 4;
        float4 v = *reinterpret_cast<const float4*>(dq + r * h + c);
        uint2 u;
        u.x = pack_bf16x2(v.x, v.y);
        u.y = pack_bf16x2(v.z, v.w);
        *reinterpret_cast<uint2*>(dqkv + r * 3 * h + c) = u;
    }
}

int encode_map3(CUtensorMap* m, const void* base, int b, int s, int cols, int64_t ld, int64_t bs) {
    uint64_t dims[3] = {(uint64_t)cols, (uint64_t)s, (uint64_t)b};
    uint64_t str[2] = {(uint64_t)ld * 2, (uint64_t)bs * 2};
    uint32_t box[3] = {64, BLK, 1};
    return cvh::encode_tmap(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, str, box, nullptr, cvh::Swizzle::B128);
}

}  // namespace

extern "C" int64_t cv_attn_bwd_workspace_bytes(int b, int heads, int head_dim, int s) {
    return (int64_t)b * s * heads * head_dim * 4 /*dq fp32*/ + (int64_t)b * heads * s * 4 /*delta*/;
}

extern "C" int cv_attn_bwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk,
                           const void* v, int64_t ldv, int64_t bsv, const void* out, const void* d_out,
                           const float* lse, void* dqkv, void* workspace, int b, int heads, int head_dim, int s,
                           int sep, float dropout_p, const uint32_t* drop_mask, void* stream) {
    CV_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "dropout probability must be in [0, 1)");
    CV_REQUIRE(dropout_p == 0.f || drop_mask != nullptr, "attention dropout needs the keep mask saved by the forward");
    CV_REQUIRE(q && k && v && out && d_out && lse && dqkv && workspace, "null pointer");
    CV_REQUIRE(head_dim == HD, "head_dim must be 64");
    CV_REQUIRE(b > 0 && heads > 0 && s > 0 && sep >= 0 && sep <= s, "bad sizes");
    CV_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && bsq % 8 == 0 && bsk % 8 == 0 && bsv % 8 == 0,
               "strides must be multiples of 8 elements");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int h = heads * HD;
    float* dq_acc = static_cast<float*>(workspace);
    float* delta = dq_acc + (size_t)b * s * h;
    CV_CUDA(cudaMemsetAsync(dq_acc, 0, (size_t)b * s * h * sizeof(float), st));
    {
        const int n = b * s * heads;
        attn_bwd_delta_kernel<<<(n + 255) / 256, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(out),
                                                              static_cast<const __nv_bfloat16*>(d_out), delta, b,
                                                              heads, s);
        CV_LAUNCH_CHECK();
    }
    alignas(64) CUtensorMap tmQ, tmK, tmV, tmDO;
    int rc;
    if ((rc = encode_map3(&tmQ, q, b, s, h, ldq, bsq))) return rc;
    if ((rc = encode_map3(&tmK, k, b, s, h, ldk, bsk))) return rc;
    if ((rc = encode_map3(&tmV, v, b, s, h, ldv, bsv))) return rc;
    if ((rc = encode_map3(&tmDO, d_out, b, s, h, h, (int64_t)s * h))) return rc;
    BwdParams p;
    p.b = b; p.heads = heads; p.s = s;
    p.sep_eff = sep;
    p.scale = 1.0f / sqrtf((float)head_dim);
    p.scale_log2 = p.scale * LOG2E;
    p.lse = lse; p.delta = delta; p.dq_acc = dq_acc;
    p.dqkv = static_cast<__nv_bfloat16*>(dqkv);
    p.drop_mask = dropout_p > 0.f ? drop_mask : nullptr;
    p.keep_rows = (s + BLK - 1) / BLK * BLK;
    p.drop_scale = dropout_p > 0.f ? 1.0f / (1.0f - dropout_p) : 1.0f;
    p.sk = s; p.kv_rows = s; p.sp_w = 1; p.sp_times = 1; p.piv_pos = nullptr; p.piv_bias_log2 = 0.f;
    static bool attr_set = false;
    if (!attr_set) {
        CV_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<MODE_DENSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        attr_set = true;
    }
    dim3 grid((s + BLK - 1) / BLK, heads, b);
    attn_bwd_kernel<MODE_DENSE><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(tmQ, tmK, tmV, tmDO, p);
    CV_LAUNCH_CHECK();
    {
        const size_t rows = (size_t)b * s;
        const size_t n4 = rows * (h / 4);
        size_t blocks = (n4 + 255) / 256;
        size_t cap = (size_t)cvh::num_sms() * 8;
        attn_bwd_dq_store_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, st>>>(
            dq_acc, static_cast<__nv_bfloat16*>(dqkv), rows, h);
        CV_LAUNCH_CHECK();
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// backward of the sparse training attention: band pass + gathered-pivot pass with the JOINT lse and
// delta = rowsum(dO o O); the pivot pass' dK / dV are scattered back to the pivot positions
// (oracle/sparse_decomposition.py: sparse_attention_two_pass_backward)
// ------------------------------------------------------------------------------------------------
namespace {
__global__ void gather_pivots_bwd_kernel(const __nv_bfloat16* __restrict__ k, int64_t ldk, int64_t bsk,
                                         const __nv_bfloat16* __restrict__ v, int64_t ldv, int64_t bsv,
                                         const int64_t* __restrict__ pos, __nv_bfloat16* __restrict__ dst,
                                         int* __restrict__ pos32, int n_piv, int h) {
    const int row = blockIdx.x;
    const int batch = row / n_piv;
    const int64_t src = pos[row];
    if (threadIdx.x == 0) pos32[row] = (int)src;
    const uint4* ks = reinterpret_cast<const uint4*>(k + (size_t)batch * bsk + (size_t)src * ldk);
    const uint4* vs = reinterpret_cast<const uint4*>(v + (size_t)batch * bsv + (size_t)src * ldv);
    uint4* d = reinterpret_cast<uint4*>(dst + (size_t)row * 2 * h);
    for (int i = threadIdx.x; i < h / 8; i += blockDim.x) {
        d[i] = ks[i];
        d[h / 8 + i] = vs[i];
    }
}

// dqkv[b, pos[p], h:3h] += dpiv[b, p, h:3h]   (pivot positions of one sequence are distinct: no atomics)
__global__ void scatter_pivot_grads_kernel(const __nv_bfloat16* __restrict__ dpiv, const int* __restrict__ pos32,
                                           __nv_bfloat16* __restrict__ dqkv, int n_piv, int s, int h) {
    const int row = blockIdx.x;
    const int batch = row / n_piv;
    const __nv_bfloat162* src = reinterpret_cast<const __nv_bfloat162*>(dpiv + (size_t)row * 3 * h + h);
    __nv_bfloat162* dst = reinterpret_cast<__nv_bfloat162*>(dqkv + ((size_t)batch * s + pos32[row]) * 3 * h + h);
    for (int i = threadIdx.x; i < h; i += blockDim.x) {          // 2h bf16 = h pairs
        const float2 a = __bfloat1622float2(dst[i]), c = __bfloat1622float2(src[i]);
        dst[i] = __floats2bfloat162_rn(a.x + c.x, a.y + c.y);
    }
}
inline size_t al256b(size_t x) { return (x + 255) / 256 * 256; }
}  // namespace

extern "C" int64_t cv_attn_sparse_bwd_workspace_bytes(int b, int heads, int head_dim, int s, int n_piv) {
    const size_t h = (size_t)heads * head_dim;
    return (int64_t)(al256b((size_t)b * s * h * 4) + al256b((size_t)b * heads * s * 4) + al256b((size_t)b * n_piv * 2 * h * 2) +
                     al256b((size_t)b * n_piv * 3 * h * 2) + al256b((size_t)b * n_piv * 4));
}

extern "C" int cv_attn_sparse_bwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk,
                                  const void* v, int64_t ldv, int64_t bsv, const int64_t* pivot_idx, const void* out,
                                  const void* d_out, const float* lse, void* dqkv, void* workspace, int b, int heads,
                                  int head_dim, int s, int n_piv, int query_window, int key_window_times,
                                  void* stream) {
    return cv_attn_sparse_dropout_bwd(q, ldq, bsq, k, ldk, bsk, v, ldv, bsv, pivot_idx, out, d_out, lse, dqkv, workspace,
                                      b, heads, head_dim, s, n_piv, query_window, key_window_times, 0.f, nullptr, stream);
}

extern "C" int cv_attn_sparse_dropout_bwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk,
                                          int64_t bsk, const void* v, int64_t ldv, int64_t bsv,
                                          const int64_t* pivot_idx, const void* out, const void* d_out,
                                          const float* lse, void* dqkv, void* workspace, int b, int heads,
                                          int head_dim, int s, int n_piv, int query_window, int key_window_times,
                                          float dropout_p, const uint32_t* drop_mask, void* stream) {
    CV_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "dropout probability must be in [0, 1)");
    CV_REQUIRE(dropout_p == 0.f || drop_mask != nullptr, "attention dropout needs the keep mask saved by the forward");
    CV_REQUIRE(q && k && v && pivot_idx && out && d_out && lse && dqkv && workspace, "null pointer");
    CV_REQUIRE(head_dim == HD, "head_dim must be 64");
    CV_REQUIRE(b > 0 && heads > 0 && s > 0 && n_piv > 0 && n_piv <= s, "bad sizes");
    CV_REQUIRE(query_window > 0 && key_window_times > 0 && s % query_window == 0,
               "the sequence length must be a multiple of query_window");
    CV_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && bsq % 8 == 0 && bsk % 8 == 0 && bsv % 8 == 0,
               "strides must be multiples of 8 elements");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int h = heads * HD;
    char* ws = static_cast<char*>(workspace);
    float* dq_acc = reinterpret_cast<float*>(ws);
    ws += al256b((size_t)b * s * h * 4);
    float* delta = reinterpret_cast<float*>(ws);
    ws += al256b((size_t)b * heads * s * 4);
    __nv_bfloat16* pkv = reinterpret_cast<__nv_bfloat16*>(ws);
    ws += al256b((size_t)b * n_piv * 2 * h * 2);
    __nv_bfloat16* dpiv = reinterpret_cast<__nv_bfloat16*>(ws);
    ws += al256b((size_t)b * n_piv * 3 * h * 2);
    int* pos32 = reinterpret_cast<int*>(ws);
    CV_CUDA(cudaMemsetAsync(dq_acc, 0, (size_t)b * s * h * sizeof(float), st));
    {
        const int n = b * s * heads;
        attn_bwd_delta_kernel<<<(n + 255) / 256, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(out),
                                                              static_cast<const __nv_bfloat16*>(d_out), delta, b,
                                                              heads, s);
        CV_LAUNCH_CHECK();
    }
    gather_pivots_bwd_kernel<<<b * n_piv, 128, 0, st>>>(static_cast<const __nv_bfloat16*>(k), ldk, bsk,
                                                       static_cast<const __nv_bfloat16*>(v), ldv, bsv, pivot_idx, pkv,
                                                       pos32, n_piv, h);
    CV_LAUNCH_CHECK();
    alignas(64) CUtensorMap tmQ, tmK, tmV, tmDO, tmPK, tmPV;
    int rc;
    if ((rc = encode_map3(&tmQ, q, b, s, h, ldq, bsq))) return rc;
    if ((rc = encode_map3(&tmK, k, b, s, h, ldk, bsk))) return rc;
    if ((rc = encode_map3(&tmV, v, b, s, h, ldv, bsv))) return rc;
    if ((rc = encode_map3(&tmDO, d_out, b, s, h, h, (int64_t)s * h))) return rc;
    if ((rc = encode_map3(&tmPK, pkv, b, n_piv, h, 2 * (int64_t)h, (int64_t)n_piv * 2 * h))) return rc;
    if ((rc = encode_map3(&tmPV, pkv + h, b, n_piv, h, 2 * (int64_t)h, (int64_t)n_piv * 2 * h))) return rc;
    BwdParams p;
    p.b = b; p.heads = heads; p.s = s;
    p.sep_eff = 0;
    p.scale = 1.0f / sqrtf((float)head_dim);
    p.scale_log2 = p.scale * LOG2E;
    p.lse = lse; p.delta = delta; p.dq_acc = dq_acc;
    // keep bits (cv_attn_sparse_drop_mask_words): band pass reads region [0], pivot pass region [1]
    const int nqb = (s + BLK - 1) / BLK, npt = (n_piv + BLK - 1) / BLK;
    const uint32_t* band_keep = dropout_p > 0.f ? drop_mask : nullptr;
    const uint32_t* piv_keep = dropout_p > 0.f ? drop_mask + (size_t)b * heads * nqb * BLK * nqb * 4 : nullptr;
    p.drop_mask = band_keep; p.keep_rows = nqb * BLK;
    p.drop_scale = dropout_p > 0.f ? 1.0f / (1.0f - dropout_p) : 1.0f;
    p.sp_w = query_window; p.sp_times = key_window_times;
    p.piv_bias_log2 = logf((float)(s / n_piv)) * LOG2E;
    static bool attr_set = false;
    if (!attr_set) {
        CV_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<MODE_BAND>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        CV_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<MODE_PIVOT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        attr_set = true;
    }
    // band pass: dK / dV rows of the sequence
    p.dqkv = static_cast<__nv_bfloat16*>(dqkv);
    p.sk = s; p.kv_rows = s; p.piv_pos = nullptr;
    attn_bwd_kernel<MODE_BAND><<<dim3((s + BLK - 1) / BLK, heads, b), NUM_THREADS, SMEM_BYTES, st>>>(tmQ, tmK, tmV, tmDO, p);
    CV_LAUNCH_CHECK();
    if (key_window_times * query_window < s) {       // some query sees pivots at all
        p.dqkv = dpiv;
        p.sk = n_piv; p.kv_rows = n_piv; p.piv_pos = pos32;
        p.drop_mask = piv_keep; p.keep_rows = npt * BLK;
        attn_bwd_kernel<MODE_PIVOT><<<dim3((n_piv + BLK - 1) / BLK, heads, b), NUM_THREADS, SMEM_BYTES, st>>>(
            tmQ, tmPK, tmPV, tmDO, p);
        CV_LAUNCH_CHECK();
        scatter_pivot_grads_kernel<<<b * n_piv, 256, 0, st>>>(dpiv, pos32, static_cast<__nv_bfloat16*>(dqkv), n_piv, s, h);
        CV_LAUNCH_CHECK();
    }
    {
        const size_t rows = (size_t)b * s;
        const size_t n4 = rows * (h / 4);
        size_t blocks = (n4 + 255) / 256;
        size_t cap = (size_t)cvh::num_sms() * 8;
        attn_bwd_dq_store_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, st>>>(
            dq_acc, static_cast<__nv_bfloat16*>(dqkv), rows, h);
        CV_LAUNCH_CHECK();
    }
    return 0;
}
