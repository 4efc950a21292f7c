// kernel='simple' with bf16 I/O (bf16 in, bf16 out; fp32 partials) -- one cooperative kernel, sm_100a.
// (fp16: pass 2 would pair an fp16 A operand with the bf16 hi/lo image of the fp32 sums in one kind::f16 MMA; the hardware
//  faulted on that mix (round 2), and an fp16 image cannot hold un-scaled sums that grow with N, so fp16 inputs are
//  up-cast and run the fp32 kernel -- ops._SimpleAttention16.)
//
// Reference path replaced: full_attention_conv(..., 'simple'), node classification/difformer.py:18-39, fed by the
// Linear outputs (`:115-118`) under bf16 / fp16 autocast.  Algorithmic bytes: read Q, K, V + write out = 4*H*D*2 =
// 2048 B per node at H = 4, D = 64 (SURVEY.md 8d): half of the fp32 path.
//
// With 16-bit inputs the operands need no CUDA-core pass at all: TMA tensor loads (cp.async.bulk.tensor.2d, 128B swizzle)
// land the [nodes][64] tiles of every head directly in the UMMA shared-memory layouts
//   pass 1  S_h = K_h^T V_h : a [32 nodes][128 B] tile IS the MN-major SW128 operand (K index = node), M = N = 128 = two
//           heads (H = 1: the two 16-node halves of the tile), one tcgen05.mma per 16 nodes -- no hi/lo split: the inputs
//           are exact 16-bit values, products and sums are exact / fp32 in TMEM;
//   pass 2  q_n (S_h | z_h)  : a [128 rows][128 B] tile IS the K-major SW128 A operand; B = the un-scaled fp32 sums split
//           into bf16 hi + lo (2 MMAs), N = 80 (64 columns of S + the z column), c = 1/(|Q||K|) applied in the epilogue.
// The only CUDA-core work of pass 1 is what has no matrix form at this size: z = sum k, u = sum v, sum k^2, sum q^2, read
// from the landed tiles by 8 warps (conflict-free swizzled LDS.128).  Tail, grid-wide / cross-GPU sum and the second grid
// barrier are shared with the fp32 kernel (simple_tc.cuh: fused_tail).
//
// Warps (12): 0 TMA issuer (both passes), 1 MMA issuer (both passes), 2-3 idle, 4-11 column sums of pass 1,
//             4-7 tail + pass-2 epilogue (TMEM lane quadrant = warp % 4).
#include <atomic>
#include <mutex>
#include <vector>

#include "simple_tc.cuh"

namespace dif {
namespace {

constexpr int kLpThreads = 12 * 32;
constexpr int kLpNodes = 32;                  // nodes per pass-1 stage
constexpr int kLpTile = kLpNodes * 128;       // one (tensor, head) tile: [32 nodes][64 x 16 bit]
constexpr int kLpNS = 4;                      // pass-1 stages
constexpr int kLpQTile = 128 * 128;           // pass 2: [128 rows][64 x 16 bit] of one head
constexpr int kLpNQ = 4;                      // pass-2 Q stages
constexpr int kLpOutBox = 32 * 128;           // per epilogue warp: [32 rows][64 x 16 bit]
constexpr int kLpOutStage = 4 * 2 * kLpOutBox;   // 4 warps x double buffer

template <int H, bool W = false>
struct LpGeo {
    static constexpr int kStage = 3 * H * kLpTile;                      // K | V | Q tiles of all heads
    static constexpr int kSmem1 = kLpNS * kStage;
    static constexpr int kSmem2 = PLay<H, W>::kBBytes + kLpNQ * kLpQTile + kLpOutStage + H * kDim * 4;
    static constexpr int kSmem = (kSmem1 > kSmem2 ? kSmem1 : kSmem2) + 1024;
    static constexpr int kChunks = H * 8;                               // 16-byte chunks per node row of one tensor
    static constexpr int kRowGroups = 256 / kChunks;                    // sum threads = 256
};

struct Bf16 {
    static constexpr int kFmt = 1;            // UMMA operand format: bf16
    __device__ static __forceinline__ void unpack2(uint32_t w, float& a, float& b) { a = __uint_as_float(w << 16); b = __uint_as_float(w & 0xffff0000u); }
    __device__ static __forceinline__ uint32_t pack2(float a, float b) { return bf2_bits(a, b); }
};

__device__ __forceinline__ uint32_t make_idesc_fmt(int M, int N, int a_mn, int b_mn, int a_fmt, int b_fmt) {
    uint32_t d = 0;
    d |= 1u << 4;                        // D format f32
    d |= (uint32_t)a_fmt << 7;           // A format: 0 = f16, 1 = bf16
    d |= (uint32_t)b_fmt << 10;
    d |= (uint32_t)a_mn << 15;           // A major: 0 = K, 1 = MN
    d |= (uint32_t)b_mn << 16;
    d |= (uint32_t)(N >> 3) << 17;
    d |= (uint32_t)(M >> 4) << 24;
    return d;
}

struct LpArgs {
    ReduceArgs1 r;            // q/k/v pointers unused (tensor maps); N, rows_per_cta, ws, flags, epoch, partials, prepared, sh, n_total, dbg
    unsigned long long* flags2;
    int store_hint, reverse, l2_hints;
};

// W ("wide"): ONE head of M = D = 128 on the H = 2 geometry (see PLay, simple_tc.cuh): the two 64-column halves of a row play the
// two heads in pass 1 (whose accumulator then is the whole S[128][128]); pass 2 contracts over K = 128 (two Q stages per tile) into
// the two output halves.
template <int H, class T, bool W = false>
__global__ void __launch_bounds__(kLpThreads, 1) simple_lp_kernel(const __grid_constant__ LpArgs la, const __grid_constant__ CUtensorMap mq,
                                                                 const __grid_constant__ CUtensorMap mk, const __grid_constant__ CUtensorMap mv,
                                                                 const __grid_constant__ CUtensorMap mo) {
    using G = Geo<H>;
    using L = LpGeo<H, W>;
    using P = PLay<H, W>;
    const ReduceArgs1& a = la.r;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    // pass 2 view
    uint8_t* Bop = base;
    uint8_t* qring = base + P::kBBytes;
    uint8_t* ostage = qring + kLpNQ * kLpQTile;
    float* us = reinterpret_cast<float*>(ostage + kLpOutStage);
    __shared__ uint64_t full[kLpNS], empty[kLpNS], done;
    __shared__ uint64_t qfull[kLpNQ], qempty[kLpNQ], tfull[kNAcc], tempty[kNAcc], bbar;
    __shared__ uint32_t tmem_slot;
    __shared__ float part[16];
    __shared__ __align__(16) float red[H == 1 ? 64 * 65 : 4096];      // [256 sum threads][z 8 | u 8]; H == 1: also the S block halves
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t r0 = (int64_t)blockIdx.x * a.rows_per_cta;
    const int64_t r1 = min(a.N, r0 + (int64_t)a.rows_per_cta);
    const int iters = r1 > r0 ? (int)((r1 - r0 + kLpNodes - 1) / kLpNodes) : 0;
    const int my_tiles = r1 > r0 ? (int)((r1 - r0 + kTile2 - 1) / kTile2) : 0;
    const int nsc = my_tiles * H;
    auto row0_of = [&](int sc) -> int64_t { const int t = sc / H; return r0 + (int64_t)(la.reverse ? my_tiles - 1 - t : t) * kTile2; };
    uint64_t* dbg = a.dbg;
    DIF_STAMP(dbg, 0);

    if (tid == 0) {
        for (int s = 0; s < kLpNS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 9); }
        for (int s = 0; s < kLpNQ; ++s) { mbar_init(&qfull[s], 1); mbar_init(&qempty[s], 1); }
        for (int s = 0; s < kNAcc; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 4); }
        mbar_init(&done, 1);
        mbar_init(&bbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    pdl_wait();                                         // programmatic dependent launch: everything above overlapped the previous kernel
    DIF_STAMP(dbg, 1);

    if (warp == 0) {
        if (lane == 0) {
            // =================== TMA issuer: pass 1 (K | V | Q tiles of every head, 32 nodes per stage) ... ===================
            const uint64_t pol_first = policy_evict_first_(), pol_last = policy_evict_last();
            const uint32_t sbase = smem_u32(base);
            for (int it = 0; it < iters; ++it) {
                const int s = it % kLpNS;
                if (it >= kLpNS) mbar_wait(&empty[s], ((it / kLpNS) - 1) & 1);
                const int row = (int)(r0 + (int64_t)it * kLpNodes);
                mbar_expect_tx(&full[s], (uint32_t)L::kStage);
                const uint32_t sb = sbase + s * L::kStage;
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    if (la.l2_hints) {
                        tma_load_2d_hint(sb + (0 * H + h) * kLpTile, &mk, h * kDim, row, &full[s], pol_first);
                        tma_load_2d_hint(sb + (1 * H + h) * kLpTile, &mv, h * kDim, row, &full[s], pol_first);
                        tma_load_2d_hint(sb + (2 * H + h) * kLpTile, &mq, h * kDim, row, &full[s], pol_last);
                    } else {
                        tma_load_2d(sb + (0 * H + h) * kLpTile, &mk, h * kDim, row, &full[s]);
                        tma_load_2d(sb + (1 * H + h) * kLpTile, &mv, h * kDim, row, &full[s]);
                        tma_load_2d(sb + (2 * H + h) * kLpTile, &mq, h * kDim, row, &full[s]);
                    }
                }
            }
            // drain: every stage that was used must have been consumed (MMA + column sums) before pass 2 re-uses the memory
            for (int it = iters; it < iters + kLpNS; ++it)
                if (it >= kLpNS) mbar_wait(&empty[it % kLpNS], ((it / kLpNS) - 1) & 1);
            // =================== ... and pass 2: Q tiles of this CTA's rows, [128 rows][128 B] per (tile, head) ===================
            const uint32_t qb = smem_u32(qring);
            const uint64_t pol_q = policy_evict_first_();
            for (int sc = 0; sc < nsc; ++sc) {
                const int s = sc % kLpNQ, h = sc % H;
                if (sc >= kLpNQ) mbar_wait(&qempty[s], ((sc / kLpNQ) - 1) & 1);
                const int row = (int)row0_of(sc);
                mbar_expect_tx(&qfull[s], (uint32_t)kLpQTile);
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    tma_load_2d_hint(qb + s * kLpQTile + i * kLpTile, &mq, h * kDim, row + i * kLpNodes, &qfull[s], pol_q);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // =================== MMA issuer: pass 1 ... ===================
            {
                const uint32_t idesc = make_idesc_fmt(128, 128, 1, 1, T::kFmt, T::kFmt);
                const uint32_t sbase = smem_u32(base);
                // H >= 2: MN blocks = the two heads of a pair (tiles kLpTile apart), two K steps of 16 nodes per stage;
                // H == 1: MN blocks = the two 16-node halves of the tile (2048 B apart), one K step
                const uint32_t lbo = H == 1 ? 2048u : (uint32_t)kLpTile, sbo = 1024;
                for (int it = 0; it < iters; ++it) {
                    const int s = it % kLpNS;
                    mbar_wait(&full[s], (it / kLpNS) & 1);
                    tc_fence_after();
                    const uint32_t sb = sbase + s * L::kStage;
#pragma unroll
                    for (int p = 0; p < G::kPairs; ++p) {
#pragma unroll
                        for (int ks = 0; ks < (H == 1 ? 1 : 2); ++ks) {
                            const uint32_t ko = (H == 1 ? 0u : (uint32_t)(2 * p) * kLpTile) + ks * 2048u;
                            const uint64_t kd = make_desc(sb + 0 * H * kLpTile + ko, lbo, sbo);
                            const uint64_t vd = make_desc(sb + 1 * H * kLpTile + ko, lbo, sbo);
                            umma(tmem + p * 128, kd, vd, idesc, (it > 0 || ks > 0) ? 1u : 0u);
                        }
                    }
                    umma_commit(&empty[s]);
                }
                if (iters > 0) umma_commit(&done); else mbar_arrive(&done);
            }
            // =================== ... and pass 2: (tile, head): 4 K steps x (q Bhi + q Blo), M = 128, N = 80 ===================
            const uint32_t idesc = make_idesc_fmt(kTile2, kBN, 0, 0, T::kFmt, 1);
            const uint32_t qb = smem_u32(qring), b_base = smem_u32(Bop);
            pdl_launch_dependents();                    // the next kernel of the stream may start its prologue as SMs free up
            mbar_wait(&bbar, 0);
            if (!W) {
                for (int sc = 0; sc < nsc; ++sc) {
                    const int s = sc % kLpNQ, slot = sc % kNAcc, h = sc % H;
                    if (sc >= kNAcc) mbar_wait(&tempty[slot], ((sc / kNAcc) - 1) & 1);
                    mbar_wait(&qfull[s], (sc / kLpNQ) & 1);
                    tc_fence_after();
                    const uint32_t sb = qb + s * kLpQTile, bb = b_base + h * 2 * kBOp;
                    const uint32_t d = tmem + slot * kAccCols;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t qd = make_desc(sb + ks * 32, kKmajLBO, kKmajSBO);
                        const uint64_t bhi = make_desc(bb + ks * 32, kKmajLBO, kKmajSBO), blo = make_desc(bb + kBOp + ks * 32, kKmajLBO, kKmajSBO);
                        umma(d, qd, bhi, idesc, ks > 0 ? 1u : 0u);
                        umma(d, qd, blo, idesc, 1u);
                    }
                    umma_commit(&qempty[s]);
                    umma_commit(&tfull[slot]);
                }
            } else {
                // wide: stage = (tile, K block kb), accumulator slot = (tile, output half dh): both K blocks feed both halves
                for (int sc = 0; sc < nsc; sc += 2) {
                    const int slot0 = sc % kNAcc, slot1 = (sc + 1) % kNAcc;
                    if (sc >= kNAcc) {
                        mbar_wait(&tempty[slot0], ((sc / kNAcc) - 1) & 1);
                        mbar_wait(&tempty[slot1], (((sc + 1) / kNAcc) - 1) & 1);
                    }
#pragma unroll
                    for (int kb = 0; kb < 2; ++kb) {
                        const int st_ = sc + kb, s = st_ % kLpNQ;
                        mbar_wait(&qfull[s], (st_ / kLpNQ) & 1);
                        tc_fence_after();
                        const uint32_t sb = qb + s * kLpQTile;
#pragma unroll
                        for (int dh = 0; dh < 2; ++dh) {
                            const uint32_t bb = b_base + (2 * dh + kb) * 2 * kBOp;
                            const uint32_t d = tmem + (dh == 0 ? slot0 : slot1) * kAccCols;
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                const uint64_t qd = make_desc(sb + ks * 32, kKmajLBO, kKmajSBO);
                                const uint64_t bhi = make_desc(bb + ks * 32, kKmajLBO, kKmajSBO), blo = make_desc(bb + kBOp + ks * 32, kKmajLBO, kKmajSBO);
                                umma(d, qd, bhi, idesc, (kb > 0 || ks > 0) ? 1u : 0u);
                                umma(d, qd, blo, idesc, 1u);
                            }
                        }
                        umma_commit(&qempty[s]);
                    }
                    umma_commit(&tfull[slot0]);
                    umma_commit(&tfull[slot1]);
                }
            }
        }
    } else if (warp >= 4) {
        // =================== pass 1: column sums z = sum k, u = sum v and the two squared norms, straight from the landed tiles ===================
        const int ts = tid - 128;                       // 256 sum threads
        const int cid = ts % L::kChunks, rg = ts / L::kChunks;
        const int hh = cid >> 3, c = cid & 7;
        float z[8], u[8], ssk = 0.f, ssq = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) { z[i] = 0.f; u[i] = 0.f; }
        {
            const uint32_t sbase = smem_u32(base);
            for (int it = 0; it < iters; ++it) {
                const int s = it % kLpNS;
                mbar_wait(&full[s], (it / kLpNS) & 1);
                const uint32_t sb = sbase + s * L::kStage;
#pragma unroll
                for (int rr = 0; rr < kLpNodes / L::kRowGroups; ++rr) {
                    const int row = rg + rr * L::kRowGroups;
                    const uint32_t off = sw128(row, c);
                    const float4 kw = lds128(sb + (0 * H + hh) * kLpTile + off);
                    const float4 vw = lds128(sb + (1 * H + hh) * kLpTile + off);
                    const float4 qw = lds128(sb + (2 * H + hh) * kLpTile + off);
                    const uint32_t kb[4] = {__float_as_uint(kw.x), __float_as_uint(kw.y), __float_as_uint(kw.z), __float_as_uint(kw.w)};
                    const uint32_t vb[4] = {__float_as_uint(vw.x), __float_as_uint(vw.y), __float_as_uint(vw.z), __float_as_uint(vw.w)};
                    const uint32_t qb4[4] = {__float_as_uint(qw.x), __float_as_uint(qw.y), __float_as_uint(qw.z), __float_as_uint(qw.w)};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float x0, x1;
                        T::unpack2(kb[j], x0, x1);
                        z[2 * j] += x0; z[2 * j + 1] += x1;
                        ssk = fmaf(x0, x0, ssk); ssk = fmaf(x1, x1, ssk);
                        T::unpack2(vb[j], x0, x1);
                        u[2 * j] += x0; u[2 * j + 1] += x1;
                        T::unpack2(qb4[j], x0, x1);
                        ssq = fmaf(x0, x0, ssq); ssq = fmaf(x1, x1, ssq);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
            }
        }
        ssk = warp_sum(ssk);
        ssq = warp_sum(ssq);
        if (lane == 0) { part[warp - 4] = ssk; part[8 + warp - 4] = ssq; }
#pragma unroll
        for (int i = 0; i < 8; ++i) { red[ts * 16 + i] = z[i]; red[ts * 16 + 8 + i] = u[i]; }
        __threadfence_block();
        if (warp >= 8) {
            bar_arrive_named(1, 256);                    // barrier A: 128 arrivals + the tail warps' sync
        } else {
            const int te = tid - 128, ew = warp - 4;     // 128 tail / epilogue threads, ew = warp % 4
            // =================== tail: record -> grid-wide (+ cross-GPU) sum -> B-operand image (simple_tc.cuh) ===================
            mbar_wait(&done, 0);
            tc_fence_after();
            bar_sync_named(1, 256);
            if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 4] = gtime();
            float* rec = a.ws + (int64_t)blockIdx.x * a.ws_len;
            for (int col = te; col < H * kDim; col += 128) {
                const int ccid = col >> 3, e = col & 7;
                float zs = 0.f, usum = 0.f;
                for (int g = 0; g < L::kRowGroups; ++g) { zs += red[(g * L::kChunks + ccid) * 16 + e]; usum += red[(g * L::kChunks + ccid) * 16 + 8 + e]; }
                rec[P::offZ + col] = zs;
                rec[P::offU + col] = usum;
            }
            if (te == 0) {
                float sk = 0.f, sq = 0.f;
                for (int w = 0; w < 8; ++w) { sk += part[w]; sq += part[8 + w]; }
                rec[P::offSq] = sq;
                rec[P::offSq + 1] = sk;
            }
            if (H == 1) bar_sync_named(2, 128);
            fused_tail<H, W>(a, la.flags2, rec, te, ew, lane, tmem, iters > 0, red);
            if (te == 0) {
                mbar_expect_tx(&bbar, (uint32_t)P::kBBytes);
                for (int i = 0; i < P::kBTiles * 2; ++i)
                    tma_load_1d(smem_u32(Bop) + i * kBOp, a.prepared + (size_t)i * kBOp, (uint32_t)kBOp, &bbar);
            }
            for (int i = te; i < H * kDim; i += 128) us[i] = __ldcg(a.partials + P::offU + i);
            const float cscale = 1.f / (sqrtf(__ldcg(a.partials + P::offSq)) * sqrtf(__ldcg(a.partials + P::offSq + 1)));
            bar_sync_named(2, 128);
            // =================== pass 2: epilogue: thread = one row; (c acc + u) / (c qz + N) -> 16-bit -> swizzled box -> TMA store ===================
            const uint32_t obox = smem_u32(ostage) + ew * 2 * kLpOutBox;
            const uint64_t pol = policy_evict_first();
            float inv_den = 0.f;
            for (int sc = 0; sc < nsc; ++sc) {
                const int64_t trow = row0_of(sc);
                const int h = sc % H, slot = sc % kNAcc;
                mbar_wait(&tfull[slot], (sc / kNAcc) & 1);
                tc_fence_after();
                const uint32_t taddr = tmem + ((uint32_t)(ew * 32) << 16) + slot * kAccCols;
                if (!W || h == 0) {          // wide: the denominator column lives in the dh = 0 accumulator and serves both halves
                    uint32_t qz_bits = tmem_ld1(taddr + kDim);
                    tmem_ld_wait1(qz_bits);
                    inv_den = 1.f / (fmaf(__uint_as_float(qz_bits), cscale, a.n_total));
                }
                const uint32_t ob = obox + (sc & 1) * kLpOutBox;
                if (lane == 0) tma_wait_read1();          // the store that used this buffer two stages ago has read it
                __syncwarp();
#pragma unroll
                for (int c0 = 0; c0 < kDim; c0 += 32) {
                    uint32_t r[32];
                    tmem_ld32(taddr + c0, r);
                    tmem_ld_wait32(r);
                    if (c0 == 32) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty[slot]);
                    }
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        uint32_t w[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float o0 = fmaf(__uint_as_float(r[j + 2 * e]), cscale, us[h * kDim + c0 + j + 2 * e]) * inv_den;
                            const float o1 = fmaf(__uint_as_float(r[j + 2 * e + 1]), cscale, us[h * kDim + c0 + j + 2 * e + 1]) * inv_den;
                            w[e] = T::pack2(o0, o1);
                        }
                        sts128(ob + sw128(lane, (c0 + j) >> 3), make_uint4(w[0], w[1], w[2], w[3]));
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    const int row = (int)trow + ew * 32;
                    if (la.store_hint) tma_store_2d_hint(&mo, ob, h * kDim, row, pol);
                    else tma_store_2d(&mo, ob, h * kDim, row);
                    tma_commit();
                }
            }
            if (lane == 0) tma_wait_all0();
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    DIF_STAMP(dbg, 7);
    if (warp == 1) tmem_dealloc(tmem, 512);
}

}  // namespace

// 16-bit [rows][cols] row-major tensor map, box = 32 rows x 64 elements (128 B), 128B swizzle; out-of-bounds rows read as
// zero and are clipped on store.  Encoded maps are cached per (base, rows, cols, type).
static int make_map16(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int fp16) {
    struct Entry { const void* b; int64_t r, c; int t; CUtensorMap m; };
    static std::mutex mu;
    static std::vector<Entry> cache;
    {
        std::lock_guard<std::mutex> lk(mu);
        for (const Entry& e : cache)
            if (e.b == base && e.r == rows && e.c == cols && e.t == fp16) { *map = e.m; return DIF_OK; }
    }
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        DIF_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q));
        DIF_REQUIRE(f && q == cudaDriverEntryPointSuccess, DIF_ECUDA, "cuTensorMapEncodeTiled not available in this driver");
        fn = (EncodeTiledFn)f;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)cols * 2};
    const cuuint32_t box[2] = {64, 32}, estr[2] = {1, 1};
    const CUresult r = fn(map, fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    DIF_REQUIRE(r == CUDA_SUCCESS, DIF_ECUDA, "cuTensorMapEncodeTiled (16-bit) failed (%d)", (int)r);
    std::lock_guard<std::mutex> lk(mu);
    if (cache.size() >= 64) cache.erase(cache.begin());
    cache.push_back(Entry{base, rows, cols, fp16, *map});
    return DIF_OK;
}

template <int H, class T, bool W = false>
static int launch_lp(const LpArgs& a, const CUtensorMap* maps, int grid, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        DIF_CUDA_OK(cudaFuncSetAttribute(simple_lp_kernel<H, T, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, LpGeo<H, W>::kSmem));
        attr_set = true;
    }
    void* args[] = {(void*)&a, (void*)&maps[0], (void*)&maps[1], (void*)&maps[2], (void*)&maps[3]};
    return launch_persistent((const void*)simple_lp_kernel<H, T, W>, grid, kLpThreads, (size_t)LpGeo<H, W>::kSmem, st, args);
}

int simple_forward_lp(const void* q, const void* k, const void* v, int dtype, int64_t N, int H, int Hv, int M, int D, double n_total,
                      float* partials, void* out, void* ws, int64_t ws_bytes, cudaStream_t st,
                      void* const* peer_bufs, int rank, int world, unsigned long long seq) {
    const bool wide = simple_wide_supported(N, H, Hv, M, D);
    DIF_REQUIRE(wide || simple_tc_supported(N, H, Hv, M, D), DIF_EUNSUPPORTED, "tcgen05 path: unsupported shape");
    DIF_REQUIRE(dtype == DIF_DTYPE_BF16, DIF_EUNSUPPORTED, "simple_forward(16-bit): bf16 only (dtype %d): up-cast fp16 and use the fp32 kernel", dtype);
    DIF_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out) & 15) == 0, DIF_EARG, "simple_forward(16-bit): q/k/v/out must be 16-byte aligned");
    DIF_REQUIRE(((uintptr_t)ws & 127) == 0, DIF_EARG, "simple_forward: workspace must be 128-byte aligned");
    DIF_REQUIRE(N < (1ll << 31), DIF_EUNSUPPORTED, "tcgen05 path: N must fit a 32-bit TMA coordinate");
    int grid;
    const int rpc = tc_rows_per_cta(N, H, &grid);
    const int64_t ws_len = wide ? PLay<2, true>::kWsLen : tc_ws_len(H);
    const int64_t poff = fused_ws_prepared_off(grid, ws_len);
    DIF_REQUIRE(ws_bytes >= poff + (wide ? (int64_t)PLay<2, true>::kBBytes : (int64_t)H * 2 * kBOp), DIF_EARG, "simple_forward: workspace too small");
    DIF_REQUIRE((((ws_len + kSlices - 1) / kSlices + 3) & ~(int64_t)3) <= 128, DIF_EUNSUPPORTED, "simple_forward: slice wider than the tail warps");
    static std::atomic<unsigned long long> epoch_src{0x5851F42D4C957F2Dull ^ (unsigned long long)(uintptr_t)&epoch_src};
    LpArgs la{};
    ReduceArgs1& a = la.r;
    a.N = N; a.rows_per_cta = rpc;
    a.ws = (float*)ws; a.ws_len = ws_len; a.flags = (unsigned long long*)((char*)ws + fused_ws_flags_off(grid, ws_len));
    la.flags2 = a.flags + (int64_t)(grid + 1) * kFlagStride;
    a.epoch = epoch_src.fetch_add(0x632BE59BD9B4E019ull) | 1ull;
    a.partials = partials; a.prepared = (uint8_t*)ws + poff;
    a.n_total = (float)n_total;
    a.sh.world = 1;
    if (peer_bufs != nullptr && world > 1) {
        DIF_REQUIRE(world <= kCommMaxRanks && rank >= 0 && rank < world && seq > 0, DIF_EARG, "simple_forward(sharded): bad rank/world/seq");
        for (int r = 0; r < world; ++r) { DIF_REQUIRE(peer_bufs[r], DIF_EARG, "simple_forward(sharded): null peer buffer"); a.sh.bufs[r] = peer_bufs[r]; }
        a.sh.rank = rank; a.sh.world = world; a.sh.seq = seq;
        a.sh.lenpad = comm_lenpad(SimpleLayout{H, Hv, M, D}.len());
        a.sh.timeout_ns = comm_timeout_ns();
    }
    static const int hints = env_int("DIF_TC_P1_HINTS", 1), sth = env_int("DIF_TC_P2_STORE_HINT", 1), rev = env_int("DIF_TC_FUSED_REVERSE", 1);
    la.l2_hints = hints; la.store_hint = sth; la.reverse = rev;
    a.dbg = dbg_buffer();
    const int fp16 = 0;
    CUtensorMap maps[4];
    int rc;
    if ((rc = make_map16(&maps[0], q, N, (int64_t)H * M, fp16))) return rc;
    if ((rc = make_map16(&maps[1], k, N, (int64_t)H * M, fp16))) return rc;
    if ((rc = make_map16(&maps[2], v, N, (int64_t)H * D, fp16))) return rc;
    if ((rc = make_map16(&maps[3], out, N, (int64_t)H * D, fp16))) return rc;
#define DIF_LP(T) (H == 4 ? launch_lp<4, T>(la, maps, grid, st) : H == 2 ? launch_lp<2, T>(la, maps, grid, st) : launch_lp<1, T>(la, maps, grid, st))
    rc = wide ? launch_lp<2, Bf16, true>(la, maps, grid, st) : DIF_LP(Bf16);
#undef DIF_LP
    if (rc) return rc;
    dbg_report("simple_lp", a.dbg, grid);
    return DIF_OK;
}

}  // namespace dif
