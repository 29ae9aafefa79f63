// cv_attn_fwd: fused dense attention forward (flash-style, nothing of size [sq, sk] ever reaches HBM).
//
// Replaces standard_attention (/root/reference/mpu/sparse_transformer.py:652-673) together with the
// split / head-permute copies around it in GPT2ParallelSelfAttention.forward (:131-163):
//     softmax( (Q / sqrt(hn)) K^T * mask - 10000 * (1 - mask) ) V
// for the two mask families the reference builds: lower-triangular (pretrain_gpt2.py:218-221) and the
// int-`sep` form (mpu/sparse_transformer.py:477-489: keys [0, sep + mem) visible to every query, causal
// after that), with sq <= sk (queries are the LAST sq positions of the sk keys: decode-with-memory prefill).
// Masked scores are exactly -10000 as in the reference; whole key tiles that are masked for every query
// of the block are skipped (their softmax weight underflows to 0 in fp32).
//
// Q, K, V are read in place from the packed QKV GEMM output [b, s, 3h] (or a KV cache) through 3-D TMA
// tensor maps; the context is written token-major [b, sq, h] — the layout the out-projection GEMM reads.
//
// One CTA per (128-query block, head, batch); 10 warps:
//   warp 0     TMA producer (Q once; K/V tiles of 128 keys through a 3-stage ring)
//   warp 1     tcgen05.mma issuer:  S = Q K^T (128x128x64) into TMEM;  O_j = P_j V_j (128x64x128) into TMEM
//   warps 2-9  softmax: two threads per query row (64 keys / 32 output dims each); tcgen05.ld S, online max/sum, P
//              (bf16) -> swizzled smem, then accumulate O_j from TMEM into registers with the running rescale
// S and O are double-buffered in TMEM so S_{j+1} is computed while the softmax of tile j runs.
#include "common.cuh"
#include "host.h"
#include "../../include/cogview_b200.h"

namespace {
using namespace cv;

constexpr int BQ = 128;       // queries per CTA
constexpr int BKV = 128;      // keys per tile
constexpr int HD = 64;        // head dim (CogView: 2560 / 40)
constexpr int KV_STAGES = 3;
constexpr int Q_BYTES = BQ * HD * 2;        // 16 KB
constexpr int K_BYTES = BKV * HD * 2;       // 16 KB
constexpr int V_BYTES = BKV * HD * 2;       // 16 KB
constexpr int P_BYTES = BQ * BKV * 2;       // 32 KB (two 128x64 K-major sub-tiles)
constexpr int SMEM_BYTES = Q_BYTES + KV_STAGES * (K_BYTES + V_BYTES) + 2 * P_BYTES + 1024 + 256 + 1024 /*sPos*/ + 6 * BQ * 4 /*sX*/;
constexpr int NUM_THREADS = 320;
constexpr float LOG2E = 1.4426950408889634f;

struct AttnParams {
    int b, heads, sq, sk;
    int sep_eff;        // keys [0, sep_eff) are visible to every query
    int off;            // sk - sq: query i sees key j <= i + off
    float scale_log2;   // (1/sqrt(hn)) * log2(e)
    __nv_bfloat16* out; // [b, sq, heads*HD]
    int64_t ldo;        // row stride of out (elements)
    int64_t bso;        // batch stride of out (elements)
    float* lse;         // [b, heads, sq] natural-log LSE, or null
    DropoutArgs drop;   // attention-probability dropout (mpu/sparse_transformer.py:667-669); p = 0 disables
    uint32_t* drop_mask;// two regions of b*heads*nkb_all*nqb_all*128 uint4 each, written by attn_dropout_mask_kernel:
                        //  [0] key-major [b, heads, nkb_all*128 (key), nqb_all, 4]: word w of (key, query block) holds
                        //      queries qb*128 + 32w .. +31 (what the backward consumes: one 16-byte load per key row)
                        //  [1] query-major [b, heads, nqb_all*128 (query), nkb_all, 4]: what this kernel consumes
    int nkb_all;        // ceil(sk / 128)
    int nqb_all;        // ceil(sq / 128)
    // sparse training attention (mpu/sparse_transformer.py:675-725; sp_w = 0: dense).  One softmax over
    //   band   : keys j with band_start(i) <= j <= i,  band_start(i) = max(0, i / sp_w - sp_times + 1) * sp_w
    //   pivots : gathered keys p with piv_pos[p] < band_start(i), score + log(s / n_piv)
    // (the closed form of the reference's window mask + rmask-gathered pivot mask, oracle/sparse_decomposition.py)
    int sp_w, sp_times, n_piv;
    const int* piv_pos;     // [b, n_piv] positions of the gathered pivot keys
    float piv_bias_log2;    // log(s / n_piv) * log2(e)
    // sparse with dropout: drop_mask holds the three regions of SparseKeepLayout instead of the two above
    int sp_npt;             // ceil(n_piv / 128): pivot tiles
    int sp_tiles;           // longest tile list of any query block (row length of the query-major region)
    const uint2* keep_q;    // start of that query-major region, as pairs of words (one 64-key half of a tile)
};

__host__ __device__ __forceinline__ int band_start(int i, int w, int times) {
    const int g = i / w - times + 1;
    return g > 0 ? g * w : 0;
}

// Tile list of query block qb in sparse mode: band tiles jb0 .. jb0 + nband - 1 of the real keys, then npt pivot tiles
// (all of them if any query of the block can see a pivot at all, else none).  Shared by the attention kernel, the
// keep-bit generator and the host, so all three walk the same list.
struct SparseTiles { int jb0, nband, npt; };
__host__ __device__ __forceinline__ SparseTiles sparse_tiles(int qb, int s, int w, int times, int n_piv) {
    const int q0 = qb * BQ;
    const int q_last = (q0 + BQ < s ? q0 + BQ : s) - 1;
    SparseTiles t;
    t.jb0 = band_start(q0, w, times) / BKV;
    t.nband = q_last / BKV - t.jb0 + 1;
    t.npt = band_start(q_last, w, times) > 0 ? (n_piv + BKV - 1) / BKV : 0;
    return t;
}

// Keep bits of the sparse attention-probability dropout (cv_attn_sparse_drop_mask_words), uint32 words:
//   [0] band key-major  at 0:        [b, heads, nqb*128 (key), nqb, 4]  — the dense key-major layout (s = sq = sk)
//   [1] pivot key-major at piv_off:  [b, heads, npt*128 (pivot slot), nqb, 4]
//   [2] query-major     at qmaj_off: [b, heads, nqb*128 (query), tiles, 4], indexed by the tile-list position j
//       (band tiles first, then pivot tiles), so the attention kernel walks it linearly
// bit i of word w of a key-major (key, query block qb) entry is query qb*128 + 32w + i; bit i of word w of a
// query-major (query, j) entry is key 32w + i of tile j.  Tiles outside a query block's list stay unwritten.
struct SparseKeepLayout { size_t piv_off, qmaj_off, words; };
__host__ __device__ __forceinline__ SparseKeepLayout sparse_keep_layout(int b, int heads, int nqb, int npt, int tiles) {
    const size_t bh = (size_t)b * heads, key_row = (size_t)nqb * 4;   // words per key row
    SparseKeepLayout l;
    l.piv_off = bh * nqb * BKV * key_row;
    l.qmaj_off = l.piv_off + bh * npt * BKV * key_row;
    l.words = l.qmaj_off + bh * nqb * BQ * (size_t)tiles * 4;
    return l;
}

template <bool DROPOUT, bool SPARSE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmPK,
                const __grid_constant__ CUtensorMap tmPV, const AttnParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sQ = smem;
    uint8_t* sKV = sQ + Q_BYTES;                              // stage s: K at s*(K+V), V after it
    uint8_t* sP = sKV + KV_STAGES * (K_BYTES + V_BYTES);      // 2 buffers
    uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * P_BYTES);
    uint64_t* q_full = bars;                 // [1]
    uint64_t* kv_full = bars + 1;            // [KV_STAGES]
    uint64_t* kv_empty = kv_full + KV_STAGES;
    uint64_t* s_full = kv_empty + KV_STAGES; // [2]
    uint64_t* p_full = s_full + 2;           // [2]
    uint64_t* o_full = p_full + 2;           // [2]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(o_full + 2);
    int* sPos = reinterpret_cast<int*>(bars + 32);           // [2][BKV] pivot positions of the current pivot tile
    float* sX = reinterpret_cast<float*>(sPos + 2 * BKV);    // [2 tiles][2 halves][BQ] row maxima, [2][BQ] row sums

    const int warp_idx = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // heaviest (last) query blocks first
    const int qb = gridDim.x - 1 - blockIdx.x;
    const int head = blockIdx.y, batch = blockIdx.z;
    const int q0 = qb * BQ;
    // number of key tiles any query of this block can see
    int kmax = q0 + BQ + p.off;              // exclusive bound of causally visible keys for the last row
    if (kmax < p.sep_eff) kmax = p.sep_eff;
    if (kmax > p.sk) kmax = p.sk;
    int nkb = (kmax + BKV - 1) / BKV;
    // sparse: band tiles jb0 .. jb0 + nband - 1 of the real keys first, then every pivot tile (if any query of the
    // block can see a pivot at all); one tile list for the three roles
    int jb0 = 0, nband = nkb;
    if (SPARSE) {
        const SparseTiles st = sparse_tiles(qb, p.sq, p.sp_w, p.sp_times, p.n_piv);
        jb0 = st.jb0;
        nband = st.nband;
        nkb = nband + st.npt;
    }

    if (warp_idx == 0 && lane == 0) {
        tma_prefetch_desc(&tmQ);
        tma_prefetch_desc(&tmK);
        tma_prefetch_desc(&tmV);
        mbar_init(q_full, 1);
        for (int i = 0; i < KV_STAGES; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&s_full[i], 1); mbar_init(&p_full[i], 256); mbar_init(&o_full[i], 1); }
        fence_barrier_init();
    }
    if (warp_idx == 1) tmem_alloc<512>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const uint32_t TM_S = 0, TM_O = 256;     // column offsets: S0, S1 (128 each); O0, O1 (64 each)

    if (warp_idx == 0) {
        if (lane == 0) {
            mbar_expect_tx(q_full, Q_BYTES);
            tma_load_3d(sQ, &tmQ, q_full, head * HD, q0, batch);
            int stage = 0; uint32_t phase = 0;
            for (int j = 0; j < nkb; ++j) {
                mbar_wait(&kv_empty[stage], phase ^ 1);
                uint8_t* sK = sKV + stage * (K_BYTES + V_BYTES);
                mbar_expect_tx(&kv_full[stage], K_BYTES + V_BYTES);
                if (SPARSE && j >= nband) {
                    tma_load_3d(sK, &tmPK, &kv_full[stage], head * HD, (j - nband) * BKV, batch);
                    tma_load_3d(sK + K_BYTES, &tmPV, &kv_full[stage], head * HD, (j - nband) * BKV, batch);
                } else {
                    tma_load_3d(sK, &tmK, &kv_full[stage], head * HD, (jb0 + j) * BKV, batch);
                    tma_load_3d(sK + K_BYTES, &tmV, &kv_full[stage], head * HD, (jb0 + j) * BKV, batch);
                }
                if (++stage == KV_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp_idx == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc_s = make_idesc_bf16(BQ, BKV, 0, 0);  // Q K-major, K K-major
            constexpr uint32_t idesc_o = make_idesc_bf16(BQ, HD, 0, 1);   // P K-major, V MN-major
            const uint32_t q_addr = smem_u32(sQ);
            auto issue_s = [&](int j, int stage) {
                const uint32_t k_addr = smem_u32(sKV + stage * (K_BYTES + V_BYTES));
#pragma unroll
                for (int k = 0; k < HD / 16; ++k) {
                    umma_f16(tmem_base + TM_S + (j & 1) * BKV, make_smem_desc_sw128(q_addr + k * 32, 0, 1024),
                             make_smem_desc_sw128(k_addr + k * 32, 0, 1024), idesc_s, k != 0);
                }
                umma_commit(&s_full[j & 1]);
            };
            mbar_wait(q_full, 0);
            int ld_stage = 0; uint32_t ld_phase = 0;   // stage/phase of the next tile whose S is issued
            mbar_wait(&kv_full[0], 0);
            tc_fence_after();
            issue_s(0, 0);
            ld_stage = 1 % KV_STAGES;
            int pv_stage = 0;
            for (int j = 0; j < nkb; ++j) {
                if (j + 1 < nkb) {
                    mbar_wait(&kv_full[ld_stage], ld_phase);
                    tc_fence_after();
                    issue_s(j + 1, ld_stage);
                    if (++ld_stage == KV_STAGES) { ld_stage = 0; ld_phase ^= 1; }
                }
                mbar_wait(&p_full[j & 1], (j >> 1) & 1);
                tc_fence_after();
                const uint32_t p_addr = smem_u32(sP + (j & 1) * P_BYTES);
                const uint32_t v_addr = smem_u32(sKV + pv_stage * (K_BYTES + V_BYTES) + K_BYTES);
#pragma unroll
                for (int k = 0; k < BKV / 16; ++k) {
                    const uint32_t pa = p_addr + (k >> 2) * (BQ * 128) + (k & 3) * 32;
                    umma_f16(tmem_base + TM_O + (j & 1) * HD, make_smem_desc_sw128(pa, 0, 1024),
                             make_smem_desc_sw128(v_addr + k * (16 * 128), BKV * 128, 1024), idesc_o, k != 0);
                }
                umma_commit(&o_full[j & 1]);
                umma_commit(&kv_empty[pv_stage]);
                if (++pv_stage == KV_STAGES) pv_stage = 0;
            }
        }
    } else {
        // ------------------------------ softmax / output warps ------------------------------
        // 8 warps: warp w works on TMEM lane quadrant w % 4 (rows 32 (w % 4) .. +31, one row per lane) and on HALF of the
        // row: warps 2-5 the first 64 keys of every tile and output dims 0-31, warps 6-9 the other half.  Two threads
        // per row halve the serial exp2 / pack / rescale chain of a tile and give every scheduler two softmax warps to
        // overlap (one warp per scheduler ran at 8 % tensor-pipe utilisation, profiles/r01_ncu_full_attention_summary);
        // the only exchange per tile is the row maximum (shared memory + a 64-thread named barrier per quadrant).
        const int q = warp_idx & 3;
        const int hf = (warp_idx - 2) >> 2;
        const int row = q * 32 + lane;
        const int qi = q0 + row;                       // query index within the sequence
        const uint32_t lane_addr = tmem_base + (uint32_t(q * 32) << 16);
        const int causal_lim = qi + p.off;             // last causally visible key
        const int bs_row = SPARSE ? band_start(qi, p.sp_w, p.sp_times) : 0;
        constexpr int HK = BKV / 2, HO = HD / 2;       // keys / output dims per thread
        float m = -INFINITY, l = 0.f, alpha_prev = 0.f;
        float o[HO];
#pragma unroll
        for (int i = 0; i < HO; ++i) o[i] = 0.f;
        const float masked_val = -10000.0f * LOG2E;
        const uint4* keep_row = nullptr;
        uint4 pre_keep = make_uint4(0u, 0u, 0u, 0u);
        uint32_t keep_off = 0u;
        if (DROPOUT && SPARSE) {
            // query-major region (p.keep_q): one row of sp_tiles entries per query, in tile-list order.  This thread
            // reads only its half's two words, after the scores are in registers (the row-maximum exchange covers the
            // load), and holds a 32-bit row offset instead of a pointer: the sparse tile walk is at the register limit
            // (168) even without dropout
            keep_off = (uint32_t)((((uint32_t)batch * p.heads + head) * p.nqb_all * BQ + qi) * p.sp_tiles * 2 + hf);
        } else if (DROPOUT) {
            const size_t region = (size_t)p.b * p.heads * p.nkb_all * p.nqb_all * (BQ * 4);   // words per region
            keep_row = reinterpret_cast<const uint4*>(p.drop_mask + region) +
                       (((size_t)batch * p.heads + head) * p.nqb_all * BQ + qi) * p.nkb_all;
            pre_keep = keep_row[0];
        }

        for (int j = 0; j < nkb; ++j) {
            uint32_t kw0 = 0u, kw1 = 0u;                // keep bits of this row over this thread's 64 keys
            if (DROPOUT && !SPARSE) {
                kw0 = hf ? pre_keep.z : pre_keep.x;
                kw1 = hf ? pre_keep.w : pre_keep.y;
                if (j + 1 < nkb) pre_keep = keep_row[j + 1];
            }
            const bool piv_tile = SPARSE && j >= nband;
            if (piv_tile) {                             // positions of this tile's 128 gathered keys -> shared memory
                if (hf == 0) {
                    const int pj = (j - nband) * BKV + row;
                    sPos[(j & 1) * BKV + row] = pj < p.n_piv ? p.piv_pos[(size_t)batch * p.n_piv + pj] : 0x7fffffff;
                }
                named_bar_sync(2, 256);
            }
            mbar_wait(&s_full[j & 1], (j >> 1) & 1);
            tc_fence_after();
            const int k0 = SPARSE ? (piv_tile ? (j - nband) * BKV : (jb0 + j) * BKV) : j * BKV;
            const int kb = k0 + hf * HK;                // first key of this thread's half
            // does this tile need per-element masking for this row?
            const bool full_vis = SPARSE ? (!piv_tile && k0 >= bs_row && k0 + BKV - 1 <= qi && k0 + BKV <= p.sk)
                                         : (k0 + BKV <= p.sk) && ((k0 + BKV <= p.sep_eff) || (k0 + BKV - 1 <= causal_lim));
            float s[HK];
#pragma unroll
            for (int c = 0; c < HK / 32; ++c) {
                uint32_t (&r)[32] = *reinterpret_cast<uint32_t(*)[32]>(&s[c * 32]);
                tmem_ld_x32(lane_addr + TM_S + (j & 1) * BKV + hf * HK + c * 32, r);
            }
            tmem_ld_wait();
            float mx = -INFINITY;
            if (full_vis) {
#pragma unroll
                for (int i = 0; i < HK; ++i) { s[i] *= p.scale_log2; mx = fmaxf(mx, s[i]); }
            } else if (piv_tile) {
                const int* pos = sPos + (j & 1) * BKV + hf * HK;
#pragma unroll
                for (int i = 0; i < HK; ++i) {
                    const int pp = pos[i];
                    float v = pp < bs_row ? s[i] * p.scale_log2 + p.piv_bias_log2 : masked_val;
                    if (pp == 0x7fffffff) v = -INFINITY;   // beyond the pivot list
                    s[i] = v;
                    mx = fmaxf(mx, v);
                }
            } else {
#pragma unroll
                for (int i = 0; i < HK; ++i) {
                    const int kj = kb + i;
                    const bool vis = SPARSE ? (kj >= bs_row && kj <= qi) : ((kj < p.sep_eff) || (kj <= causal_lim));
                    float v = vis ? s[i] * p.scale_log2 : masked_val;
                    if (kj >= p.sk) v = -INFINITY;     // key does not exist
                    s[i] = v;
                    mx = fmaxf(mx, v);
                }
            }
            if (DROPOUT && SPARSE) {
                const uint2 kw = p.keep_q[keep_off + j * 2];
                kw0 = kw.x;
                kw1 = kw.y;
            }
            // row maximum over both halves
            sX[((j & 1) * 2 + hf) * BQ + row] = mx;
            named_bar_sync(3 + q, 64);
            mx = fmaxf(fmaxf(mx, sX[((j & 1) * 2 + (hf ^ 1)) * BQ + row]), m);
            const float alpha = exp2f(m - mx);          // m = -inf on the first tile -> 0
            m = mx;
            float psum = 0.f;
            uint8_t* prow = sP + (j & 1) * P_BYTES + hf * (BQ * 128) + row * 128;   // this half = one 64-key sub-tile
#pragma unroll
            for (int c = 0; c < HK / 8; ++c) {          // 8 chunks of 8 keys (16 bytes)
                float e[8];
#pragma unroll
                for (int t = 0; t < 8; ++t) e[t] = exp2f(s[c * 8 + t] - mx);
                uint4 pk;
                pk.x = pack_bf16x2(e[0], e[1]); pk.y = pack_bf16x2(e[2], e[3]);
                pk.z = pack_bf16x2(e[4], e[5]); pk.w = pack_bf16x2(e[6], e[7]);
                // the row sum uses the bf16-rounded probabilities that the PV MMA will see
                const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&pk);
#pragma unroll
                for (int t = 0; t < 4; ++t) psum += __low2float(pb[t]) + __high2float(pb[t]);
                if (DROPOUT && SPARSE) {   // as below, on the packed words (bf16 zero = 0x0000): e[] is dead here
                    const uint32_t w = ((c >> 2) == 0 ? kw0 : kw1) >> ((c & 3) * 8);
                    pk.x &= ((w & 1u) ? 0x0000FFFFu : 0u) | ((w & 2u) ? 0xFFFF0000u : 0u);
                    pk.y &= ((w & 4u) ? 0x0000FFFFu : 0u) | ((w & 8u) ? 0xFFFF0000u : 0u);
                    pk.z &= ((w & 16u) ? 0x0000FFFFu : 0u) | ((w & 32u) ? 0xFFFF0000u : 0u);
                    pk.w &= ((w & 64u) ? 0x0000FFFFu : 0u) | ((w & 128u) ? 0xFFFF0000u : 0u);
                } else if (DROPOUT) {   // dropout acts on the normalised probabilities: the row sum stays undropped;
                                        // the 1/(1-p) scale is applied once to the output row at the end
                    const uint32_t w = (c >> 2) == 0 ? kw0 : kw1;
#pragma unroll
                    for (int t = 0; t < 8; ++t) e[t] = ((w >> ((c & 3) * 8 + t)) & 1u) ? e[t] : 0.f;
                    pk.x = pack_bf16x2(e[0], e[1]); pk.y = pack_bf16x2(e[2], e[3]);
                    pk.z = pack_bf16x2(e[4], e[5]); pk.w = pack_bf16x2(e[6], e[7]);
                }
                *reinterpret_cast<uint4*>(prow + ((c ^ (row & 7)) << 4)) = pk;
            }
            l = l * alpha + psum;                       // this half's share of the row sum
            fence_proxy_async_smem();
            tc_fence_before();
            mbar_arrive(&p_full[j & 1]);
            if (j > 0) {
                mbar_wait(&o_full[(j - 1) & 1], ((j - 1) >> 1) & 1);
                tc_fence_after();
                uint32_t r[HO];
                tmem_ld_x32(lane_addr + TM_O + ((j - 1) & 1) * HD + hf * HO, r);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < HO; ++i) o[i] = o[i] * alpha_prev + __uint_as_float(r[i]);
            }
            alpha_prev = alpha;
        }
        {
            const int j = nkb - 1;
            mbar_wait(&o_full[j & 1], (j >> 1) & 1);
            tc_fence_after();
            uint32_t r[HO];
            tmem_ld_x32(lane_addr + TM_O + (j & 1) * HD + hf * HO, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < HO; ++i) o[i] = o[i] * alpha_prev + __uint_as_float(r[i]);
        }
        // total row sum = the two halves' shares
        sX[(4 + hf) * BQ + row] = l;
        named_bar_sync(3 + q, 64);
        l += sX[(4 + (hf ^ 1)) * BQ + row];
        if (qi < p.sq) {
            const float inv_l = (DROPOUT ? p.drop.scale : 1.0f) / l;
            __nv_bfloat16* orow = p.out + (size_t)batch * p.bso + (size_t)qi * p.ldo + head * HD + hf * HO;
#pragma unroll
            for (int c = 0; c < HO / 8; ++c) {
                uint4 pk;
                pk.x = pack_bf16x2(o[c * 8 + 0] * inv_l, o[c * 8 + 1] * inv_l);
                pk.y = pack_bf16x2(o[c * 8 + 2] * inv_l, o[c * 8 + 3] * inv_l);
                pk.z = pack_bf16x2(o[c * 8 + 4] * inv_l, o[c * 8 + 5] * inv_l);
                pk.w = pack_bf16x2(o[c * 8 + 6] * inv_l, o[c * 8 + 7] * inv_l);
                *reinterpret_cast<uint4*>(orow + c * 8) = pk;
            }
            if (hf == 0 && p.lse != nullptr)
                p.lse[((size_t)batch * p.heads + head) * p.sq + qi] = m * 0.6931471805599453f + logf(l);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp_idx == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

// Keep decisions of the attention-probability dropout for every (query, key) pair of the visible tiles, generated
// ahead of the attention kernel at full occupancy (inside the attention kernel the same work sits on the softmax
// warps' critical path: measured +200 us per call at the 4B shape).  One thread per (query row, key tile): a
// Philox4x32-10 call seeds four 32-step LCG streams, keep iff state >= p * 2^32.  Writes both layouts (AttnParams).
// SPARSE: blockIdx.y is the position j in the block's tile list (sparse_tiles) and the three regions of
// SparseKeepLayout are written.  A band tile keeps its key-tile index as counter, pivot tile t counts as key tile
// nkb_all + t: the pivot slots and the band keys of one query draw from disjoint counters.  Either way every decision
// is a pure function of (seed, site, batch, head, query, key or pivot slot), which checkpoint recomputation relies on.
template <bool SPARSE>
__global__ void __launch_bounds__(128, SPARSE ? 3 : 4)   // sparse: a few more live values; 3 blocks / SM keep it spill-free
attn_dropout_mask_kernel(const AttnParams p) {
    const int qb = blockIdx.x, j = blockIdx.y;
    const int head = blockIdx.z % p.heads, batch = blockIdx.z / p.heads;
    const int q0 = qb * BQ;
    int ctile = j;                               // counter tile: the key tile, or nkb_all + pivot tile
    if (SPARSE) {
        const SparseTiles st = sparse_tiles(qb, p.sq, p.sp_w, p.sp_times, p.n_piv);
        if (j >= st.nband + st.npt) return;      // beyond this block's tile list
        ctile = j < st.nband ? st.jb0 + j : p.nkb_all + (j - st.nband);
    } else {
        int kmax = q0 + BQ + p.off;
        if (kmax < p.sep_eff) kmax = p.sep_eff;
        if (kmax > p.sk) kmax = p.sk;
        if (j * BKV >= kmax) return;             // tile never visited by the attention kernels
    }
    const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
    const int qi = q0 + threadIdx.x;
    const int ctr_tiles = SPARSE ? p.nkb_all + p.sp_npt : p.nkb_all;
    const uint64_t ctr = (((uint64_t)batch * p.heads + head) * p.sq + qi) * ctr_tiles + ctile;
    const uint4 r0 = philox4x32_10(p.drop.seed, ctr, p.drop.stream);
    uint32_t rng[4] = {r0.x, r0.y, r0.z, r0.w};
    uint32_t wrow[4], wkey[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        uint32_t bits = 0u, mine = 0u;
#pragma unroll
        for (int t = 0; t < 32; ++t) {
            rng[g] = rng[g] * 1664525u + 1013904223u;
            const bool keep = rng[g] >= p.drop.threshold;
            bits |= (keep ? 1u : 0u) << t;
            const uint32_t bal = __ballot_sync(0xffffffffu, keep);   // key 32g + t over this warp's 32 queries
            if (lane == t) mine = bal;
        }
        wrow[g] = bits;
        wkey[g] = mine;
    }
    const size_t bh = (size_t)batch * p.heads + head;
    uint32_t* dm;
    if (SPARSE) {
        const SparseKeepLayout l = sparse_keep_layout(p.b, p.heads, p.nqb_all, p.sp_npt, p.sp_tiles);
        reinterpret_cast<uint4*>(p.drop_mask + l.qmaj_off)[(bh * p.nqb_all * BQ + qi) * p.sp_tiles + j] =
            make_uint4(wrow[0], wrow[1], wrow[2], wrow[3]);
        dm = ctile < p.nkb_all
                 ? p.drop_mask + ((bh * p.nkb_all * BKV + ctile * BKV + lane) * p.nqb_all + qb) * 4 + wq
                 : p.drop_mask + l.piv_off +
                       ((bh * p.sp_npt * BKV + (ctile - p.nkb_all) * BKV + lane) * p.nqb_all + qb) * 4 + wq;
    } else {
        const size_t region = (size_t)p.b * p.heads * p.nkb_all * p.nqb_all * (BQ * 4);
        reinterpret_cast<uint4*>(p.drop_mask + region)[(bh * p.nqb_all * BQ + qi) * p.nkb_all + j] =
            make_uint4(wrow[0], wrow[1], wrow[2], wrow[3]);
        dm = p.drop_mask + ((bh * p.nkb_all * BKV + j * BKV + lane) * p.nqb_all + qb) * 4 + wq;
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) dm[(size_t)g * 32 * p.nqb_all * 4] = wkey[g];
}

// [b, s, cols] bf16 view: row stride ld, batch stride bs (elements); box [64 cols x box_rows rows x 1]
int encode_qkv_map(CUtensorMap* m, const void* base, int b, int s, int cols, int64_t ld, int64_t bs, int box_rows) {
    uint64_t dims[3] = {(uint64_t)cols, (uint64_t)s, (uint64_t)b};
    uint64_t str[2] = {(uint64_t)ld * 2, (uint64_t)bs * 2};
    uint32_t box[3] = {64, (uint32_t)box_rows, 1};
    return cvh::encode_tmap(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, str, box, nullptr, cvh::Swizzle::B128);
}

}  // namespace

extern "C" int cv_attn_fwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk,
                           const void* v, int64_t ldv, int64_t bsv, void* out, int64_t ldo, int64_t bso, float* lse,
                           int b, int heads, int head_dim, int sq, int sk, int sep, float dropout_p, uint64_t seed,
                           uint32_t site, uint32_t* drop_mask, void* stream) {
    CV_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "dropout probability must be in [0, 1)");
    CV_REQUIRE(dropout_p == 0.f || drop_mask != nullptr, "attention dropout needs the keep-mask buffer");
    CV_REQUIRE(q && k && v && out, "null pointer");
    CV_REQUIRE(head_dim == HD, "head_dim must be 64 (CogView: hidden / heads = 64)");
    CV_REQUIRE(b > 0 && heads > 0 && sq > 0 && sk >= sq, "need sk >= sq > 0");
    CV_REQUIRE(sep >= 0 && sep <= sq, "sep must be in [0, sq]");
    CV_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0 && bsq % 8 == 0 && bsk % 8 == 0 &&
                   bsv % 8 == 0 && bso % 8 == 0,
               "strides must be multiples of 8 elements");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    alignas(64) CUtensorMap tmQ, tmK, tmV;
    int rc;
    if ((rc = encode_qkv_map(&tmQ, q, b, sq, heads * HD, ldq, bsq, BQ))) return rc;
    if ((rc = encode_qkv_map(&tmK, k, b, sk, heads * HD, ldk, bsk, BKV))) return rc;
    if ((rc = encode_qkv_map(&tmV, v, b, sk, heads * HD, ldv, bsv, BKV))) return rc;
    AttnParams p;
    p.b = b; p.heads = heads; p.sq = sq; p.sk = sk;
    p.off = sk - sq;
    p.sep_eff = sep > 0 ? sep + (sk - sq) : 0;   // mpu/sparse_transformer.py:486; sep = 0 with memory: see below
    // NB: with sep == 0 the reference still marks the memory columns [0, sk - sq) visible (:486 with sep = 0);
    // they are causally visible anyway (j <= i + off for every i >= 0), so sep_eff = 0 is equivalent.
    p.scale_log2 = (1.0f / sqrtf((float)head_dim)) * LOG2E;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.ldo = ldo; p.bso = bso;
    p.lse = lse;
    {
        const cvh::HostDropout hd = cvh::make_dropout(dropout_p, seed, site);
        p.drop.p = hd.p; p.drop.scale = hd.scale; p.drop.threshold = hd.threshold; p.drop.stream = hd.stream;
        p.drop.seed = hd.seed;
        p.drop_mask = drop_mask;
        p.nkb_all = (sk + BKV - 1) / BKV;
        p.nqb_all = (sq + BQ - 1) / BQ;
    }
    p.sp_w = 0; p.sp_times = 0; p.n_piv = 0; p.piv_pos = nullptr; p.piv_bias_log2 = 0.f;
    p.sp_npt = 0; p.sp_tiles = 0; p.keep_q = nullptr;
    static bool attr_set = false;
    if (!attr_set) {
        CV_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        CV_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        attr_set = true;
    }
    dim3 grid((sq + BQ - 1) / BQ, heads, b);
    if (dropout_p > 0.f) {
        attn_dropout_mask_kernel<false><<<dim3(p.nqb_all, p.nkb_all, b * heads), 128, 0, s>>>(p);
        CV_LAUNCH_CHECK();
        attn_fwd_kernel<true, false><<<grid, NUM_THREADS, SMEM_BYTES, s>>>(tmQ, tmK, tmV, tmK, tmV, p);
    }
    else attn_fwd_kernel<false, false><<<grid, NUM_THREADS, SMEM_BYTES, s>>>(tmQ, tmK, tmV, tmK, tmV, p);
    CV_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// sparse training attention (mpu/sparse_transformer.py:675-725): gathered pivots + causal band, one softmax
// ------------------------------------------------------------------------------------------------
namespace {
// gathered pivot keys / values: dst[b, p, 0:h] = K[b, pos[p], :], dst[b, p, h:2h] = V[b, pos[p], :]; pos32 = (int)pos
__global__ void gather_pivots_kernel(const __nv_bfloat16* __restrict__ k, int64_t ldk, int64_t bsk,
                                     const __nv_bfloat16* __restrict__ v, int64_t ldv, int64_t bsv,
                                     const int64_t* __restrict__ pos, __nv_bfloat16* __restrict__ dst,
                                     int* __restrict__ pos32, int b, int n_piv, int h) {
    const int row = blockIdx.x;                 // (batch, pivot)
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

// longest sparse tile list over the query blocks (row length of the query-major keep-bit region)
int sparse_max_tiles(int s, int w, int times, int n_piv) {
    int m = 0;
    for (int qb = 0; qb < (s + BQ - 1) / BQ; ++qb) {
        const SparseTiles t = sparse_tiles(qb, s, w, times, n_piv);
        m = std::max(m, t.nband + t.npt);
    }
    return m;
}
}  // namespace

extern "C" int64_t cv_attn_sparse_workspace_bytes(int b, int heads, int head_dim, int n_piv) {
    const int64_t h = (int64_t)heads * head_dim;
    return ((int64_t)b * n_piv * 2 * h * 2 + 255) / 256 * 256 + (int64_t)b * n_piv * 4;
}

extern "C" int64_t cv_attn_sparse_drop_mask_words(int b, int heads, int s, int n_piv, int query_window,
                                                  int key_window_times) {
    if (b <= 0 || heads <= 0 || s <= 0 || n_piv <= 0 || query_window <= 0 || key_window_times <= 0) return 0;
    const int nqb = (s + BQ - 1) / BQ, npt = (n_piv + BKV - 1) / BKV;
    return (int64_t)sparse_keep_layout(b, heads, nqb, npt, sparse_max_tiles(s, query_window, key_window_times, n_piv))
        .words;
}

extern "C" int cv_attn_sparse_fwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk,
                                  const void* v, int64_t ldv, int64_t bsv, const int64_t* pivot_idx, void* out,
                                  int64_t ldo, int64_t bso, float* lse, void* workspace, int b, int heads,
                                  int head_dim, int s, int n_piv, int query_window, int key_window_times,
                                  void* stream) {
    return cv_attn_sparse_dropout_fwd(q, ldq, bsq, k, ldk, bsk, v, ldv, bsv, pivot_idx, out, ldo, bso, lse, workspace, b,
                                      heads, head_dim, s, n_piv, query_window, key_window_times, 0.f, 0, 0, nullptr,
                                      stream);
}

extern "C" int cv_attn_sparse_dropout_fwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk,
                                          int64_t bsk, const void* v, int64_t ldv, int64_t bsv,
                                          const int64_t* pivot_idx, void* out, int64_t ldo, int64_t bso, float* lse,
                                          void* workspace, int b, int heads, int head_dim, int s, int n_piv,
                                          int query_window, int key_window_times, float dropout_p, uint64_t seed,
                                          uint32_t site, uint32_t* drop_mask, void* stream) {
    CV_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "dropout probability must be in [0, 1)");
    CV_REQUIRE(dropout_p == 0.f || drop_mask != nullptr, "attention dropout needs the keep-mask buffer");
    CV_REQUIRE(q && k && v && pivot_idx && out && workspace, "null pointer");
    CV_REQUIRE(head_dim == HD, "head_dim must be 64 (CogView: hidden / heads = 64)");
    CV_REQUIRE(b > 0 && heads > 0 && s > 0 && n_piv > 0 && n_piv <= s, "bad sizes");
    CV_REQUIRE(query_window > 0 && key_window_times > 0 && s % query_window == 0,
               "the sequence length must be a multiple of query_window (mpu/sparse_transformer.py:703,713)");
    CV_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0 && bsq % 8 == 0 && bsk % 8 == 0 &&
                   bsv % 8 == 0 && bso % 8 == 0,
               "strides must be multiples of 8 elements");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int h = heads * HD;
    __nv_bfloat16* pkv = static_cast<__nv_bfloat16*>(workspace);
    int* pos32 = reinterpret_cast<int*>(static_cast<char*>(workspace) + ((size_t)b * n_piv * 2 * h * 2 + 255) / 256 * 256);
    gather_pivots_kernel<<<b * n_piv, 128, 0, st>>>(static_cast<const __nv_bfloat16*>(k), ldk, bsk,
                                                   static_cast<const __nv_bfloat16*>(v), ldv, bsv, pivot_idx, pkv, pos32,
                                                   b, n_piv, h);
    CV_LAUNCH_CHECK();
    alignas(64) CUtensorMap tmQ, tmK, tmV, tmPK, tmPV;
    int rc;
    if ((rc = encode_qkv_map(&tmQ, q, b, s, h, ldq, bsq, BQ))) return rc;
    if ((rc = encode_qkv_map(&tmK, k, b, s, h, ldk, bsk, BKV))) return rc;
    if ((rc = encode_qkv_map(&tmV, v, b, s, h, ldv, bsv, BKV))) return rc;
    if ((rc = encode_qkv_map(&tmPK, pkv, b, n_piv, h, 2 * (int64_t)h, (int64_t)n_piv * 2 * h, BKV))) return rc;
    if ((rc = encode_qkv_map(&tmPV, pkv + h, b, n_piv, h, 2 * (int64_t)h, (int64_t)n_piv * 2 * h, BKV))) return rc;
    AttnParams p;
    p.b = b; p.heads = heads; p.sq = s; p.sk = s;
    p.off = 0; p.sep_eff = 0;
    p.scale_log2 = (1.0f / sqrtf((float)head_dim)) * LOG2E;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.ldo = ldo; p.bso = bso; p.lse = lse;
    p.drop.p = 0.f; p.drop.scale = 1.f; p.drop.threshold = 0; p.drop.stream = 0; p.drop.seed = 0;
    p.drop_mask = nullptr;
    p.nkb_all = (s + BKV - 1) / BKV;
    p.nqb_all = (s + BQ - 1) / BQ;
    p.sp_w = query_window; p.sp_times = key_window_times; p.n_piv = n_piv; p.piv_pos = pos32;
    p.piv_bias_log2 = logf((float)(s / n_piv)) * LOG2E;           // integer division as in :697
    p.sp_npt = (n_piv + BKV - 1) / BKV;
    p.sp_tiles = 0; p.keep_q = nullptr;
    dim3 grid((s + BQ - 1) / BQ, heads, b);
    if (dropout_p > 0.f) {
        static bool attr_set_drop = false;
        if (!attr_set_drop) {
            CV_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         SMEM_BYTES));
            attr_set_drop = true;
        }
        const cvh::HostDropout hd = cvh::make_dropout(dropout_p, seed, site);
        p.drop.p = hd.p; p.drop.scale = hd.scale; p.drop.threshold = hd.threshold; p.drop.stream = hd.stream;
        p.drop.seed = hd.seed;
        p.drop_mask = drop_mask;
        p.sp_tiles = sparse_max_tiles(s, query_window, key_window_times, n_piv);
        CV_REQUIRE((int64_t)b * heads * p.nqb_all * BQ * p.sp_tiles * 2 < (int64_t(1) << 32),
                   "batch x heads x sequence too large for the sparse attention keep bits");
        p.keep_q = reinterpret_cast<const uint2*>(
            drop_mask + sparse_keep_layout(b, heads, p.nqb_all, p.sp_npt, p.sp_tiles).qmaj_off);
        attn_dropout_mask_kernel<true><<<dim3(p.nqb_all, p.sp_tiles, b * heads), 128, 0, st>>>(p);
        CV_LAUNCH_CHECK();
        attn_fwd_kernel<true, true><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(tmQ, tmK, tmV, tmPK, tmPV, p);
    } else {
        static bool attr_set = false;
        if (!attr_set) {
            CV_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         SMEM_BYTES));
            attr_set = true;
        }
        attn_fwd_kernel<false, true><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(tmQ, tmK, tmV, tmPK, tmPV, p);
    }
    CV_LAUNCH_CHECK();
    return 0;
}
