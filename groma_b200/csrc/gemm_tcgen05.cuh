// Persistent, warp-specialised bf16 GEMM for sm_100a:  D[M,N] = sum_taps A[M + off(tap), K] * B[N, tap*K + K]^T
//   - operands are K-major bf16 in HBM, moved by TMA (128B swizzle) into a multi-stage shared-memory ring
//   - one elected thread issues tcgen05.mma (cta_group::1, M=128, N=BN, K=16), fp32 accumulators live in TMEM
//   - two TMEM accumulator stages so the epilogue of tile i overlaps the MMAs of tile i+1
//   - 4 epilogue warps: tcgen05.ld -> bias / activation / LayerScale / residual -> bf16|fp32 stores
// "taps" turn the same kernel into an implicit-GEMM 3x3 convolution over zero-bordered flat NHWC maps
// (each tap is a row shift of A and a K offset of B), see DESIGN.md "conv as shifted-row GEMM".
#pragma once
#include "ptx.cuh"
#include "decode_common.cuh"

namespace gb {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_MAX_TAPS = 27;
constexpr int GEMM_THREADS = 192;  // warp0 TMA, warp1 MMA, warps 2..5 epilogue (tiles narrower than 128 columns)
// Wide tiles (BN >= 128) run EIGHT epilogue warps: two per TMEM lane quarter, each draining half of the tile's columns.  With one
// epilogue warp per SM sub-partition the 128 x 256 tile of a K = 1024 GEMM (ViT) took longer to drain (bias + erf-GELU + pack +
// store ~ 9 k cycles) than its 16 k-blocks take on the tensor pipe (8 k cycles): 43.7 % tensor-active (profiles/r01_gemm_k1024_AFTER.md).
__host__ __device__ constexpr int gemm_epi_warps(int bn) { return bn >= 128 ? 8 : 4; }
__host__ __device__ constexpr int gemm_threads(int bn) { return 64 + 32 * gemm_epi_warps(bn); }

enum GemmAct : int { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2, ACT_SWIGLU = 3 };
enum GemmFlags : int {
    GF_OUT_F32 = 1,       // out is fp32 (else bf16)
    GF_BIAS_ALONG_M = 2,  // bias/gamma indexed by row (swap-AB calls)
    GF_PARTIAL = 4,       // store raw fp32 accumulators to ws[split][m][n] (split-K / deferred epilogue)
    GF_CONV_ROWS = 8,     // rows are pixels of zero-bordered [img][hp][wp] maps: skip border rows
    GF_CONV_COMPACT = 16, // with GF_CONV_ROWS: write row index of the un-padded [img][h][w] layout
    GF_PDL = 64,          // launched with programmatic stream serialisation: A (weights) is prefetched before griddepcontrol.wait,
                          // and the dependent grid is released at kernel start (it parks at its own griddepcontrol.wait)
    GF_PARTIAL_T = 128,   // with GF_PARTIAL: partials stored transposed, ws[split][n][m] (swap-AB decode: token-major rows)
    GF_ROPE_QKV = 256,    // fused LLaMA qkv projection: rotate q/k (RoPE) in the epilogue, q -> out, k/v -> the KV cache (256-wide tiles, D = 128)
};

struct GemmParams {
    CUtensorMap tma_a;  // [rows_a, K_total_a] bf16, box {64, 128}
    CUtensorMap tma_b;  // [N, taps*K]        bf16, box {64, BN}
    int M, N, K;        // K = reduction length per tap
    int num_taps;
    int a_row_off[GEMM_MAX_TAPS];  // row shift of A per tap (may be negative: TMA zero-fills OOB)
    int split_k;                   // >=1; >1 requires GF_PARTIAL
    int flags;
    int act;
    void* out;            // bf16 or fp32
    long long ld_m, ld_n;  // element strides of out / residual
    const float* bias;     // fp32 [N] (or [M]) or null
    const float* gamma;    // fp32 LayerScale [N] (or [M]) or null: v *= gamma before residual
    const __nv_bfloat16* residual;  // same strides as out, or null
    float* ws;             // fp32 partials [split][M][N] when GF_PARTIAL
    int conv_hp, conv_wp;  // padded map dims for GF_CONV_ROWS
    // GF_ROPE_QKV: rows = (sequence b, token t) with t < rope_T; columns = [q | k | v] x [rope_H heads] x [128]
    const float* rope_cos;  // fp32 [max_pos, 64]
    const float* rope_sin;
    __nv_bfloat16* rope_k;  // KV cache [B, rope_H, rope_cap, 128]
    __nv_bfloat16* rope_v;
    int rope_T, rope_H, rope_pos0;
    long long rope_cap;
};

template <int BN, int CG = 1>
struct GemmCfg {
    static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;
    static constexpr int B_ROWS = BN / CG;             // cta_group::2: each CTA of the pair stages half of the B tile
    static constexpr int B_BYTES = B_ROWS * GEMM_BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
#ifndef GROMA_BN16_STAGES
#define GROMA_BN16_STAGES 4
#endif
    static constexpr int STAGES = (CG == 2) ? 6 : ((BN >= 256) ? 4 : (BN >= 128 ? 6 : (BN == 16 ? GROMA_BN16_STAGES : 8)));
    static constexpr int TMEM_COLS = (2 * BN < 32) ? 32 : 2 * BN;
    static constexpr int EPW = gemm_epi_warps(BN);
    static constexpr int THREADS = gemm_threads(BN);
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + EPW * (32 * 80 + 32 * 8) /*epilogue staging*/ +
                                      EPW * 1024 /*per-warp bias | gamma of the tile's columns*/;
};

// Grouped rasterisation: consecutive tiles walk GROUP_M m-blocks before advancing n, so the ~148 tiles in flight share
// ~16 A row-blocks and ~9 B column-blocks -- both stay L2-resident instead of re-streaming B (180 MB for the 22016-wide
// gate/up projection) once per 1.7 m-blocks as a plain n-fastest order did (measured 939 -> see profiles/).
__device__ __forceinline__ void tile_coords(int tile, int m_tiles, int n_tiles, int& m_blk, int& n_blk) {
    constexpr int GROUP_M = 16;
    const int per_group = GROUP_M * n_tiles;
    const int g = tile / per_group;
    const int first_m = g * GROUP_M;
    const int gsize = min(GROUP_M, m_tiles - first_m);
    const int r = tile - g * per_group;
    m_blk = first_m + r % gsize;
    n_blk = r / gsize;
}

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == ACT_GELU) return gelu_erf(v);
    if (act == ACT_RELU) return fmaxf(v, 0.0f);
    return v;
}

// CG = 1: one CTA per 128 x BN tile (cta_group::1).  CG = 2: a 2-CTA cluster computes a 256 x BN tile with
// tcgen05.mma.cta_group::2 -- each CTA stages its own 128 rows of A and HALF of the B tile, the pair's tensor cores read
// both halves, so shared-memory fill + operand-read traffic per SM drops from ~192 to ~128 B/clk (the limiter of the
// single-CTA 128x256 tile) and the ring deepens from 4 to 6 stages.  Leader CTA (rank 0) issues the MMAs; barriers:
// full (leader, one arrive per CTA + all TMA bytes), empty / tmem_full (both CTAs, multicast commit), tmem_empty (leader).
template <int BN, int CG>
__global__ void __launch_bounds__(gemm_threads(BN), 1) gemm_bf16_tcgen05_kernel(const __grid_constant__ GemmParams p) {
    using Cfg = GemmCfg<BN, CG>;
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;   // [2]
    uint64_t* tempty_bar = tfull_bar + 2;       // [2]
    uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    constexpr int STG_WARP_BYTES = 32 * 80 + 32 * 8;  // 32 rows x (64 B + 16 B pad) + 32 output-row indices
    uint8_t* stage_base = reinterpret_cast<uint8_t*>(tmem_holder + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    const int crank = (CG == 2) ? (int)cluster_ctarank() : 0;     // rank inside the CTA pair
    const int wid0 = blockIdx.x / CG, wstride = gridDim.x / CG;     // work is distributed over clusters
    const int m_tiles = (p.M + GEMM_BM * CG - 1) / (GEMM_BM * CG);  // cluster-level m blocks (128*CG rows)
    const int n_tiles = (p.N + BN - 1) / BN;
    const int kb_per_tap = (p.K + GEMM_BK - 1) / GEMM_BK;
    const int total_iters = kb_per_tap * p.num_taps;
    const int iters_per_split = (total_iters + p.split_k - 1) / p.split_k;
    const int num_work = m_tiles * n_tiles * p.split_k;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tma_a);
        tma_prefetch_desc(&p.tma_b);
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int i = 0; i < STAGES; ++i) {
                mbar_init(&full_bar[i], CG);   // one arrive per CTA of the pair (+ the TMA bytes of both)
                mbar_init(&empty_bar[i], 1);
            }
            for (int i = 0; i < 2; ++i) {
                mbar_init(&tfull_bar[i], 1);
                mbar_init(&tempty_bar[i], Cfg::EPW * CG);  // one arrive per epilogue warp (of both CTAs)
            }
            fence_barrier_init();
        }
        __syncwarp();
        if constexpr (CG == 2) tmem_alloc_2cta<Cfg::TMEM_COLS>(tmem_holder);
        else tmem_alloc<Cfg::TMEM_COLS>(tmem_holder);
    }
    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    // Dependents only touch this grid's results after their own griddepcontrol.wait (= this grid complete and flushed), so
    // releasing them now is safe; it lets the next kernels become resident and the next GEMM stream its weights early.
    if (p.flags & GF_PDL) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            // work iterator over this CTA's (work item, k-iteration) pairs
            int w = wid0, it = 0, it1 = 0, m_blk = 0, n_blk = 0;
            auto load_work = [&]() {
                while (w < num_work) {
                    const int split = w % p.split_k;
                    const int tile = w / p.split_k;
                    tile_coords(tile, m_tiles, n_tiles, m_blk, n_blk);
                    m_blk = m_blk * CG + crank;           // this CTA's 128-row block
                    it = split * iters_per_split;
                    it1 = min(total_iters, it + iters_per_split);
                    if (it < it1) return true;
                    w += wstride;   // empty split: nothing to load
                }
                return false;
            };
            bool have = load_work();
            if ((CG == 1) && (p.flags & GF_PDL)) {
                // The A operand (weights) does not depend on the previous kernel: fill the ring with A tiles first, only then
                // wait for the producer of B (activations).  Hides launch + prologue + first-byte latency of every decode GEMM.
                int bc0[STAGES], bc1[STAGES];
                int issued = 0;
                while (have && issued < STAGES) {
                    const int tap = it / kb_per_tap, kb = it - tap * kb_per_tap;
                    mbar_expect_tx(&full_bar[issued], Cfg::STAGE_BYTES);
                    tma_load_2d(smem + issued * Cfg::STAGE_BYTES, &p.tma_a, &full_bar[issued], kb * GEMM_BK, m_blk * GEMM_BM + p.a_row_off[tap]);
                    bc0[issued] = tap * p.K + kb * GEMM_BK;
                    bc1[issued] = n_blk * BN;
                    ++issued;
                    if (++it >= it1) { w += wstride; have = load_work(); }
                }
                asm volatile("griddepcontrol.wait;" ::: "memory");
                for (int i = 0; i < issued; ++i)
                    tma_load_2d(smem + i * Cfg::STAGE_BYTES + Cfg::A_BYTES, &p.tma_b, &full_bar[i], bc0[i], bc1[i]);
                if (issued == STAGES) { stage = 0; phase = 1; } else { stage = issued; }
            }
            while (have) {
                const int tap = it / kb_per_tap, kb = it - tap * kb_per_tap;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                uint8_t* sb = sa + Cfg::A_BYTES;
                const int c0 = kb * GEMM_BK, c1 = m_blk * GEMM_BM + p.a_row_off[tap];
                if constexpr (CG == 2) {
                    // both CTAs credit the LEADER's full barrier: the leader arms it with the bytes of the whole pair
                    if (crank == 0) mbar_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
                    else mbar_arrive_cta(&full_bar[stage], 0);
                    tma_load_2d_2sm(sa, &p.tma_a, &full_bar[stage], c0, c1);
                    tma_load_2d_2sm(sb, &p.tma_b, &full_bar[stage], tap * p.K + kb * GEMM_BK, n_blk * BN + crank * Cfg::B_ROWS);
                } else {
                    mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                    tma_load_2d(sa, &p.tma_a, &full_bar[stage], c0, c1);
                    tma_load_2d(sb, &p.tma_b, &full_bar[stage], tap * p.K + kb * GEMM_BK, n_blk * BN);
                }
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
                if (++it >= it1) { w += wstride; have = load_work(); }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0 && crank == 0) {          // cta_group::2: only the leader CTA issues MMAs
            constexpr uint32_t idesc = make_idesc_bf16(GEMM_BM * CG, BN);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int w = wid0; w < num_work; w += wstride) {
                const int split = w % p.split_k;
                const int it0 = split * iters_per_split;
                const int it1 = min(total_iters, it0 + iters_per_split);
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int it = it0; it < it1; ++it) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
                    const uint32_t sb = sa + Cfg::A_BYTES;
                    const uint64_t da = make_sw128_kmajor_desc(sa);
                    const uint64_t db = make_sw128_kmajor_desc(sb);
#pragma unroll
                    for (int k = 0; k < GEMM_BK / 16; ++k) {
                        // advancing 16 bf16 (=32 B) along K inside the swizzle atom: +2 in 16-byte units
                        if constexpr (CG == 2) umma_bf16_2cta(d_tmem, da + 2 * k, db + 2 * k, idesc, (it > it0 || k > 0) ? 1u : 0u);
                        else umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (it > it0 || k > 0) ? 1u : 0u);
                    }
                    if constexpr (CG == 2) umma_commit_2cta(&empty_bar[stage], 0x3); else umma_commit(&empty_bar[stage]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if constexpr (CG == 2) umma_commit_2cta(&tfull_bar[acc], 0x3); else umma_commit(&tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue warps (2..5, and 6..9 on wide tiles) =====================
        const int q = warp & 3;  // TMEM lane quarter this warp may access
        constexpr int EPH = Cfg::EPW / 4;                 // warps sharing a lane quarter: each drains BN / EPH columns
        const int col_lo = ((warp - 2) >> 2) * (BN / EPH), col_hi = col_lo + BN / EPH;
        int acc = 0;
        uint32_t acc_phase = 0;
        const bool out_f32 = (p.flags & GF_OUT_F32) != 0;
        const bool bias_m = (p.flags & GF_BIAS_ALONG_M) != 0;
        const bool partial = (p.flags & GF_PARTIAL) != 0;
        for (int w = wid0; w < num_work; w += wstride) {
            const int split = w % p.split_k;
            const int tile = w / p.split_k;
            int m_blk, n_blk;
            tile_coords(tile, m_tiles, n_tiles, m_blk, n_blk);
            m_blk = m_blk * CG + crank;
            const int it0 = split * iters_per_split;
            const bool has_work = it0 < total_iters;  // an empty split contributes zeros
            const int row = m_blk * GEMM_BM + q * 32 + lane;
            bool row_ok = row < p.M;
            long long out_row = row;
            if (p.flags & GF_CONV_ROWS) {
                const int per_img = p.conv_hp * p.conv_wp;
                const int img = row / per_img, rem = row - img * per_img;
                const int y = rem / p.conv_wp, x = rem - y * p.conv_wp;
                row_ok = row_ok && y >= 1 && y <= p.conv_hp - 2 && x >= 1 && x <= p.conv_wp - 2;
                if (p.flags & GF_CONV_COMPACT)
                    out_row = (long long)img * (p.conv_hp - 2) * (p.conv_wp - 2) + (long long)(y - 1) * (p.conv_wp - 2) + (x - 1);
            }
            constexpr int CHUNK = (BN >= 32) ? 32 : 16;
            // bf16 row-major outputs go through a warp-private shared-memory transpose so that global stores are
            // sector-complete and coalesced (4 lanes x 16 B per 64-byte row segment) instead of 32 scattered 16-byte writes
            const bool staged = !partial && !out_f32 && p.ld_n == 1 && (p.ld_m & 7) == 0 &&
                                (reinterpret_cast<uintptr_t>(p.out) & 15) == 0;
            uint8_t* stg = stage_base + (warp - 2) * STG_WARP_BYTES;
            long long* stg_rows = reinterpret_cast<long long*>(stg + 32 * 80);
            if (staged) stg_rows[lane] = row_ok ? out_row : -1;
            const uint32_t stg_s = smem_u32(stg);
            bool released = false;
            int c_first = col_lo;
            // The bias / LayerScale values of this warp's columns are fetched ONCE per tile (one float4 of each per lane, while
            // the tile's MMAs are still running) into a per-warp kilobyte of shared memory and read back as broadcast LDS.  As
            // per-chunk global loads (8 + 8 LDG.128 per 32 columns) they missed the ~28 KB of L1 left beside 220 KB of shared memory
            // -- the residual / output stream evicts them -- and every chunk paid a chain of L2 round trips.
            const uint32_t bg_s = smem_u32(stage_base + Cfg::EPW * STG_WARP_BYTES + (warp - 2) * 1024);
            const bool use_bg = !bias_m && !partial && (p.bias != nullptr || p.gamma != nullptr);
            if (use_bg) {
                __syncwarp();   // the previous tile's readers are done with the buffer
                const int c = lane * 4;
                if (c < BN / EPH) {
                    const int n = n_blk * BN + col_lo + c;
                    float b4[4] = {0.f, 0.f, 0.f, 0.f}, g4[4] = {1.f, 1.f, 1.f, 1.f};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (p.bias != nullptr && n + u < p.N) b4[u] = __ldg(p.bias + n + u);
                        if (p.gamma != nullptr && n + u < p.N) g4[u] = __ldg(p.gamma + n + u);
                    }
                    st_shared_v4(bg_s + c * 4, make_uint4(__float_as_uint(b4[0]), __float_as_uint(b4[1]), __float_as_uint(b4[2]), __float_as_uint(b4[3])));
                    st_shared_v4(bg_s + 512 + c * 4, make_uint4(__float_as_uint(g4[0]), __float_as_uint(g4[1]), __float_as_uint(g4[2]), __float_as_uint(g4[3])));
                }
                __syncwarp();
            }
            // While the tile's MMAs are still running: pull this lane's residual row segment (BN / EPH columns) towards L2, so
            // the epilogue's residual loads are L2 hits instead of exposed DRAM round trips (the short-K ViT projections spent
            // their epilogue in stall_long_sb on exactly these loads)
            if (p.residual != nullptr && !partial && p.ld_n == 1 && row_ok) {
                const char* rp = reinterpret_cast<const char*>(p.residual + out_row * p.ld_m + (long long)n_blk * BN + col_lo);
#pragma unroll
                for (int b = 0; b < (BN / EPH) * 2; b += 128)
                    if (n_blk * BN + col_lo + (b >> 1) < p.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + b));
            }
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            if constexpr (BN == 256 && Cfg::EPW == 8) {
                if (p.flags & GF_ROPE_QKV) {
                    // This warp's 128 columns are exactly one head of q, k or v.  The projection is rounded to bf16 first (what the
                    // unfused path stored before rope_kv_kernel re-read it), q/k are rotated in fp32 with the pair (j, j + 64)
                    // ($HF/models/llama/modeling_llama.py:138-168), and the row goes straight to q_out / the KV cache: the
                    // [B*T, 3*H*D] intermediate and its second pass over HBM are gone.
                    c_first = col_hi;
                    const int nh = n_blk * BN + col_lo;
                    const int HD = p.rope_H << 7;
                    const int which = nh / HD;                       // 0 = q, 1 = k, 2 = v
                    const int head = (nh - which * HD) >> 7;
                    const int bb = row / p.rope_T, tt = row - bb * p.rope_T;
                    const int pos = p.rope_pos0 + tt;
                    __nv_bfloat16* dst = (which == 0)
                        ? reinterpret_cast<__nv_bfloat16*>(p.out) + (long long)row * HD + (head << 7)
                        : (which == 1 ? p.rope_k : p.rope_v) + ((((long long)bb * p.rope_H + head) * p.rope_cap + pos) << 7);
                    const float* cs = p.rope_cos + (long long)pos * 64;
                    const float* sn = p.rope_sin + (long long)pos * 64;
#pragma unroll 1
                    for (int cc = 0; cc < 2; ++cc) {
                        uint32_t v1[32], v2[32];
                        const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * BN + col_lo + 32 * cc);
                        __syncwarp();
                        tmem_ld32(taddr, v1);
                        tmem_ld32(taddr + 64, v2);
                        tmem_ld_wait();
                        if (!row_ok || nh >= p.N) continue;
                        uint32_t o1[16], o2[16];
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            float x1[4], x2[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                x1[u] = __bfloat162float(__float2bfloat16_rn(__uint_as_float(v1[j + u])));
                                x2[u] = __bfloat162float(__float2bfloat16_rn(__uint_as_float(v2[j + u])));
                            }
                            __nv_bfloat16 r1[4], r2[4];
                            if (which < 2) {
                                const float4 c4 = *reinterpret_cast<const float4*>(cs + 32 * cc + j);
                                const float4 s4 = *reinterpret_cast<const float4*>(sn + 32 * cc + j);
                                rope_pair(x1[0], x2[0], c4.x, s4.x, r1[0], r2[0]);
                                rope_pair(x1[1], x2[1], c4.y, s4.y, r1[1], r2[1]);
                                rope_pair(x1[2], x2[2], c4.z, s4.z, r1[2], r2[2]);
                                rope_pair(x1[3], x2[3], c4.w, s4.w, r1[3], r2[3]);
                            } else {
#pragma unroll
                                for (int u = 0; u < 4; ++u) { r1[u] = __float2bfloat16_rn(x1[u]); r2[u] = __float2bfloat16_rn(x2[u]); }
                            }
                            o1[j >> 1] = (uint32_t)__bfloat16_as_ushort(r1[0]) | ((uint32_t)__bfloat16_as_ushort(r1[1]) << 16);
                            o1[(j >> 1) + 1] = (uint32_t)__bfloat16_as_ushort(r1[2]) | ((uint32_t)__bfloat16_as_ushort(r1[3]) << 16);
                            o2[j >> 1] = (uint32_t)__bfloat16_as_ushort(r2[0]) | ((uint32_t)__bfloat16_as_ushort(r2[1]) << 16);
                            o2[(j >> 1) + 1] = (uint32_t)__bfloat16_as_ushort(r2[2]) | ((uint32_t)__bfloat16_as_ushort(r2[3]) << 16);
                        }
#pragma unroll
                        for (int j = 0; j < 16; j += 4) {
                            *reinterpret_cast<uint4*>(dst + 32 * cc + 2 * j) = make_uint4(o1[j], o1[j + 1], o1[j + 2], o1[j + 3]);
                            *reinterpret_cast<uint4*>(dst + 64 + 32 * cc + 2 * j) = make_uint4(o2[j], o2[j + 1], o2[j + 2], o2[j + 3]);
                        }
                    }
                }
            }
            // The residual row segment of a chunk is requested BEFORE its accumulators are read (the two latencies overlap),
            // and the accumulator stage goes back to the MMA warp as soon as the last chunk sits in registers, not after it has
            // been stored.  (Double-buffering the tcgen05.ld across chunks was tried as well: the 32 extra registers pushed
            // loop invariants into local memory, and with ~28 KB of L1 those reloads are L2 round trips -- ncu showed every
            // long-scoreboard stall of the epilogue on them; profiles/r02_gemm_epilogue_v2.md.)
            const uint32_t tbase = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * BN);
            const bool res_vec_ok = p.residual != nullptr && !partial && p.ld_n == 1 && (p.ld_m & 7) == 0;
#pragma unroll 1
            for (int c0 = c_first; c0 < col_hi; c0 += CHUNK) {
                uint32_t v[32];
                const int n0 = n_blk * BN + c0;
                const bool active = row_ok && n0 < p.N;
                uint4 rpre[4];
                const bool res_pre = res_vec_ok && active && CHUNK == 32 && n0 + CHUNK <= p.N;
                if (res_pre) {
                    const __nv_bfloat16* r = p.residual + out_row * p.ld_m + n0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) rpre[j] = __ldg(reinterpret_cast<const uint4*>(r) + j);
                }
                __syncwarp();  // tcgen05.ld is .sync.aligned (and orders the staging buffer reuse)
                if (CHUNK == 32) tmem_ld32(tbase + c0, v); else tmem_ld16(tbase + c0, v);
                tmem_ld_wait();
                if (c0 + CHUNK >= col_hi) {
                    // every column of this warp's share is in registers: release the accumulator stage now
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) { if constexpr (CG == 2) mbar_arrive_cta(&tempty_bar[acc], 0); else mbar_arrive(&tempty_bar[acc]); }
                    released = true;
                }
                if (!staged && !active) continue;
                if (!has_work) {
#pragma unroll
                    for (int j = 0; j < CHUNK; ++j) v[j] = 0u;
                }
                if (partial && (p.flags & GF_PARTIAL_T)) {
                    // lanes = consecutive rows m -> each store instruction writes 128 contiguous bytes of ws[split][n][:]
                    float* dst = p.ws + ((long long)split * p.N + n0) * p.M + out_row;
                    _Pragma("unroll") for (int j = 0; j < CHUNK; ++j) if (n0 + j < p.N) dst[(long long)j * p.M] = __uint_as_float(v[j]);
                    continue;
                }
                if (partial) {
                    float* dst = p.ws + ((long long)split * p.M + out_row) * p.N + n0;
                    if ((p.N & 3) == 0 && n0 + CHUNK <= p.N) {
#pragma unroll
                        for (int j = 0; j < CHUNK; j += 4)
                            *reinterpret_cast<uint4*>(dst + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                    } else {
                        _Pragma("unroll") for (int j = 0; j < CHUNK; ++j) if (n0 + j < p.N) dst[j] = __uint_as_float(v[j]);
                    }
                    continue;
                }
                // ---- full epilogue: bias -> act -> gamma -> residual
                const bool swiglu = p.act == ACT_SWIGLU;
                const int out_cols = swiglu ? CHUNK / 2 : CHUNK;
                const int no0 = swiglu ? (n0 >> 1) : n0;
                const int NO = swiglu ? (p.N >> 1) : p.N;
                float f[32];
                if (active) {
                    // every runtime switch is hoisted out of the per-element loops (one predicated branch per chunk, not per
                    // element: the first version spent its time in instruction-cache misses, see profiles/r01_gemm_epilogue.md)
                    const bool full = n0 + CHUNK <= p.N;
#pragma unroll
                    for (int j = 0; j < CHUNK; ++j) f[j] = __uint_as_float(v[j]);
                    if (p.bias) {
                        if (bias_m) {
                            const float bm = p.bias[row];
#pragma unroll
                            for (int j = 0; j < CHUNK; ++j) f[j] += bm;
                        } else if (use_bg) {
#pragma unroll
                            for (int j = 0; j < CHUNK; j += 4) {
                                const uint4 b4 = ld_shared_v4(bg_s + (c0 - col_lo + j) * 4);
                                f[j] += __uint_as_float(b4.x); f[j + 1] += __uint_as_float(b4.y);
                                f[j + 2] += __uint_as_float(b4.z); f[j + 3] += __uint_as_float(b4.w);
                            }
                        } else if (full) {
#pragma unroll
                            for (int j = 0; j < CHUNK; j += 4) {
                                const float4 b4 = *reinterpret_cast<const float4*>(p.bias + n0 + j);
                                f[j] += b4.x; f[j + 1] += b4.y; f[j + 2] += b4.z; f[j + 3] += b4.w;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < CHUNK; ++j) if (n0 + j < p.N) f[j] += p.bias[n0 + j];
                        }
                    }
                    if (swiglu) {
                        // columns (2j, 2j+1) = (gate_j, up_j): out[:, n/2] = silu(gate) * up
#pragma unroll
                        for (int j = 0; j < CHUNK / 2; ++j) f[j] = silu(f[2 * j]) * f[2 * j + 1];
                    } else {
                        if (p.act == ACT_GELU) {
#pragma unroll
                            for (int j = 0; j < CHUNK; ++j) f[j] = gelu_erf(f[j]);
                        } else if (p.act == ACT_RELU) {
#pragma unroll
                            for (int j = 0; j < CHUNK; ++j) f[j] = fmaxf(f[j], 0.0f);
                        }
                        if (p.gamma) {
                            if (bias_m) {
                                const float gm = p.gamma[row];
#pragma unroll
                                for (int j = 0; j < CHUNK; ++j) f[j] *= gm;
                            } else if (use_bg) {
#pragma unroll
                                for (int j = 0; j < CHUNK; j += 4) {
                                    const uint4 g4 = ld_shared_v4(bg_s + 512 + (c0 - col_lo + j) * 4);
                                    f[j] *= __uint_as_float(g4.x); f[j + 1] *= __uint_as_float(g4.y);
                                    f[j + 2] *= __uint_as_float(g4.z); f[j + 3] *= __uint_as_float(g4.w);
                                }
                            } else if (full) {
#pragma unroll
                                for (int j = 0; j < CHUNK; j += 4) {
                                    const float4 g4 = *reinterpret_cast<const float4*>(p.gamma + n0 + j);
                                    f[j] *= g4.x; f[j + 1] *= g4.y; f[j + 2] *= g4.z; f[j + 3] *= g4.w;
                                }
                            } else {
#pragma unroll
                                for (int j = 0; j < CHUNK; ++j) if (n0 + j < p.N) f[j] *= p.gamma[n0 + j];
                            }
                        }
                        if (p.residual) {
                            const __nv_bfloat16* r = p.residual + out_row * p.ld_m + (long long)n0 * p.ld_n;
                            if (p.ld_n == 1 && (p.ld_m & 7) == 0 && full) {
#pragma unroll
                                for (int j = 0; j < CHUNK; j += 8) {
                                    const uint4 rv = res_pre ? rpre[(j >> 3) & 3] : *reinterpret_cast<const uint4*>(r + j);
                                    const __nv_bfloat162* r2 = reinterpret_cast<const __nv_bfloat162*>(&rv);
#pragma unroll
                                    for (int t = 0; t < 4; ++t) {
                                        const float2 rf = __bfloat1622float2(r2[t]);
                                        f[j + 2 * t] += rf.x;
                                        f[j + 2 * t + 1] += rf.y;
                                    }
                                }
                            } else {
                                _Pragma("unroll") for (int j = 0; j < CHUNK; ++j) if (n0 + j < p.N) f[j] += __bfloat162float(r[(long long)j * p.ld_n]);
                            }
                        }
                    }
                }
                if (staged && CHUNK == 32 && !swiglu && n0 + CHUNK <= p.N) {
                    // 32 rows x 64 B through shared memory: 4 x STS.128 (own row), 4 x LDS.128 (4 lanes per row, 8 rows per
                    // instruction), 4 x STG.128 writing 8 complete 64-byte row segments each -- no generic-address accesses and
                    // no load -> branch -> load -> store chain per slot
                    if (active) {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            st_shared_v4(stg_s + lane * 80 + j * 16,
                                         make_uint4(pack_bf16x2(f[8 * j], f[8 * j + 1]), pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                                                    pack_bf16x2(f[8 * j + 4], f[8 * j + 5]), pack_bf16x2(f[8 * j + 6], f[8 * j + 7])));
                    }
                    __syncwarp();
                    uint4 val[4];
                    long long orow_k[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        orow_k[k] = ld_shared_b64(stg_s + 32 * 80 + (k * 8 + (lane >> 2)) * 8);
                        val[k] = ld_shared_v4(stg_s + (k * 8 + (lane >> 2)) * 80 + (lane & 3) * 16);
                    }
                    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(p.out) + n0 + (lane & 3) * 8;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (orow_k[k] >= 0) *reinterpret_cast<uint4*>(ob + orow_k[k] * p.ld_m) = val[k];
                    continue;
                }
                if (staged) {
                    const int pitch = out_cols * 2 + 16;  // +16 B: conflict-free 16-byte row writes
                    if (active) {
                        uint4* srow = reinterpret_cast<uint4*>(stg + lane * pitch);
#pragma unroll
                        for (int j = 0; j < CHUNK; j += 8)
                            if (j < out_cols)
                                srow[j >> 3] = make_uint4(pack_bf16x2(f[j], f[j + 1]), pack_bf16x2(f[j + 2], f[j + 3]),
                                                          pack_bf16x2(f[j + 4], f[j + 5]), pack_bf16x2(f[j + 6], f[j + 7]));
                    }
                    __syncwarp();
                    const int lpr = out_cols >> 3;       // lanes per output row (16 B each)
                    const int rpi = 32 / lpr;            // rows per store instruction
                    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(p.out);
                    for (int k = 0; k < lpr; ++k) {
                        const int rr = k * rpi + lane / lpr, cc = lane % lpr;
                        const long long orow = stg_rows[rr];
                        const int col = no0 + cc * 8;
                        if (orow >= 0 && col < NO) {
                            const uint4 val = *reinterpret_cast<const uint4*>(stg + rr * pitch + cc * 16);
                            __nv_bfloat16* dst = ob + orow * p.ld_m + col;
                            if (col + 8 <= NO) {
                                *reinterpret_cast<uint4*>(dst) = val;
                            } else {
                                const __nv_bfloat16* hv = reinterpret_cast<const __nv_bfloat16*>(&val);
                                for (int t = 0; t < 8 && col + t < NO; ++t) dst[t] = hv[t];
                            }
                        }
                    }
                    continue;
                }
                // ---- direct (unstaged) stores: fp32 outputs, strided / unaligned outputs
                const long long obase = out_row * p.ld_m + (long long)no0 * p.ld_n;
                if (out_f32) {
                    float* dst = reinterpret_cast<float*>(p.out) + obase;
                    if (p.ld_n == 1 && (p.ld_m & 3) == 0 && (no0 & 3) == 0 && no0 + CHUNK <= NO && !swiglu) {
#pragma unroll
                        for (int j = 0; j < CHUNK; j += 4)
                            *reinterpret_cast<float4*>(dst + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                    } else {
                        _Pragma("unroll") for (int j = 0; j < CHUNK; ++j) if (j < out_cols && no0 + j < NO) dst[(long long)j * p.ld_n] = f[j];
                    }
                } else {
                    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + obase;
                    _Pragma("unroll") for (int j = 0; j < CHUNK; ++j) if (j < out_cols && no0 + j < NO) dst[(long long)j * p.ld_n] = __float2bfloat16_rn(f[j]);
                }
            }
            // release this accumulator stage back to the MMA warp (of the leader CTA)
            if (!released) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { if constexpr (CG == 2) mbar_arrive_cta(&tempty_bar[acc], 0); else mbar_arrive(&tempty_bar[acc]); }
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();   // pair: no CTA may exit while its peer still signals its barriers
    if (warp == 1) {
        tc_fence_after();
        if constexpr (CG == 2) tmem_dealloc_2cta<Cfg::TMEM_COLS>(tmem_base);
        else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
    }
}

}  // namespace gb
