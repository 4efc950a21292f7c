// kernel='simple' -- tcgen05 / TMEM / TMA path for sm_100a (H in {1, 2, 4}, M = D = 64, fp32 in / fp32 out).
//
// Reference path replaced: full_attention_conv(..., 'simple'), node classification/difformer.py:18-39.
//
// Both contractions of the O(N) kernel run on the 5th-gen tensor cores:
//   pass 1  S_h  = K_h^T V_h      contraction over NODES  -> operands MN-major, M = N = 128 (two heads
//                                  stacked; the two diagonal 64x64 blocks of D are S_{2p}, S_{2p+1})
//   pass 2  q_n (c S_h | c z_h)   contraction over m      -> operands K-major, M = 128 rows, N = 80
//                                  (64 columns of S plus the z column = the denominator)
// Inputs are fp32; the reference tolerance (1e-3, also on the intermediates) rules out TF32
// (truncation bias ~1e-3), so every fp32 value x is split on the fly into bf16 hi + bf16 lo
// (x = hi + lo + O(2^-17 x)) and each product uses 3 MMAs (hi*hi + hi*lo + lo*hi), error ~2^-16.
// The split runs on the CUDA cores of the warps that stream the rows from HBM (256-bit loads),
// which write the bf16 tiles straight into the 128B-swizzled UMMA layout in shared memory;
// an elected thread issues tcgen05.mma with the accumulators in TMEM; mbarrier rings couple
// producers -> MMA -> epilogue.  The tensor pipe needs ~20% of the HBM time, so the kernels are
// HBM-bound by design (roofline: 4*H*D*4 B per node, SURVEY.md 8d).
//
// Pass 1 (reduce_tma_kernel<H>, 10 warps, cooperative launch, 1 CTA/SM, contiguous row range per CTA):
//   warp 8   TMA issuer: cp.async.bulk of the stage's K | V | Q rows into an fp32 staging ring (3 stages)
//   warps 0-7 converters: LDS.128 -> bf16 hi/lo split -> swizzled MN-major UMMA operand ring (+ sum k, sum v, sum k^2, sum q^2)
//   warp 9   MMA issuer (one thread): M = N = 128 (two 64-wide blocks: two heads, or two node halves when H = 1), K = 16
//   tail     TMEM -> per-CTA record, flag publish, fused deterministic cross-CTA (and cross-GPU) slice sum, pass-2 operand image
// Pass 2 (apply_tc_kernel<H,SHARED>, 13 warps, persistent over 128-row tiles):
//   warps 0-7 Q producers (LDG.256 -> bf16 hi/lo -> K-major SW128), warps 8-11 epilogue (tcgen05.ld -> (c acc + u)/(c qz + N)
//   -> swizzled staging -> TMA tensor store), warp 12 MMA issuer.
// Pass 2 with the layer epilogue (layer_tc_kernel<H,SHARED>, 17 warps): the same with 8 epilogue warps, two threads per output row.
#include <stdlib.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "simple_tc.cuh"

namespace dif {

int simple_finalize_fwd(const float* ws, int nchunks, int H, int Hv, int M, int D, float* partials, cudaStream_t st);

namespace {

// BWD = false: forward pass 1 (S = K^T V, z, u, norms).
// BWD = true : backward pass 1 (SURVEY.md 8a-1b): dS = Q^T dnum, dz = sum q dden, du = sum dnum, t_q, with
//              den = c q.z + N, dnum = g/den, dden = -(g.out)/den computed per (node, head) from the staged rows.
template <int H, bool BWD>
__global__ void __launch_bounds__(kThreadsT, 1) reduce_tma_kernel(const __grid_constant__ ReduceArgs1 a) {
    using G = Geo<H>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* stg = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* ops = stg + G::kNSG * G::kStg;
    __shared__ uint64_t sfull[G::kNSG], sempty[G::kNSG], ofull[G::kNO], oempty[G::kNO], done, tail_bar;
    __shared__ uint32_t tmem_slot;
    __shared__ float part[16];
    __shared__ __align__(16) float szc[BWD ? H * kDim : 4], su[BWD ? H * kDim : 4];   // BWD: c*z[h][m], u[h][d]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t r0 = (int64_t)blockIdx.x * a.rows_per_cta;
    const int64_t r1 = min(a.N, r0 + (int64_t)a.rows_per_cta);
    const int iters = r1 > r0 ? (int)((r1 - r0 + G::kNodes - 1) / G::kNodes) : 0;
    uint64_t* dbg = a.dbg;
    DIF_STAMP(dbg, 0);
    if (BWD) {
        const float c = 1.f / (sqrtf(a.fwd_partials[G::offSq]) * sqrtf(a.fwd_partials[G::offSq + 1]));
        for (int i = tid; i < H * kDim; i += kThreadsT) { szc[i] = a.fwd_partials[G::offZ + i] * c; su[i] = a.fwd_partials[G::offU + i]; }
    }

    if (tid == 0) {
        for (int s = 0; s < G::kNSG; ++s) { mbar_init(&sfull[s], 1); mbar_init(&sempty[s], 8); }
        for (int s = 0; s < G::kNO; ++s) { mbar_init(&ofull[s], 8); mbar_init(&oempty[s], 1); }
        mbar_init(&done, 1);
        mbar_init(&tail_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 9) tmem_alloc(&tmem_slot, G::kTmemCols1);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    DIF_STAMP(dbg, 1);

    // a converter thread always sees the same 4 columns: column chunk (tid mod 16H) of every row it touches
    float zacc[4] = {0.f, 0.f, 0.f, 0.f}, uacc[4] = {0.f, 0.f, 0.f, 0.f};
    float ssk = 0.f, ssq = 0.f;

    if (warp < 8) {
        // ===== converters: thread t handles 16-byte chunks u = t + 256 i (i < kBlocks) of each staged tensor
        const uint32_t stg_base = smem_u32(stg), ops_base = smem_u32(ops);
        for (int it = 0; it < iters; ++it) {
            const int s = it % G::kNSG, o = it % G::kNO;
            const int nrows = (int)min((int64_t)G::kNodes, r1 - (r0 + (int64_t)it * G::kNodes));
            mbar_wait(&sfull[s], (it / G::kNSG) & 1);
            if (it == 0) DIF_STAMP(dbg, 2);
            float4 x[G::kChunksPerThread][3];
#pragma unroll
            for (int i = 0; i < G::kChunksPerThread; ++i) {
                const int u = tid + 256 * i, node = u / G::kChunksPerRow;
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    x[i][t] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (node < nrows && (t == 0 || BWD || !a.gram)) x[i][t] = lds128(stg_base + s * G::kStg + t * G::kStgT + u * 16);
                }
            }
            if (!BWD && H > 1 && a.vbar != nullptr) {
                // mean_h V for the fused layer's gcn term (the head mean commutes with the SpMM): thread t -> (node t>>4,
                // 4 columns t&15); the H head chunks of that (node, columns) are read back from the fp32 staging row
                const int node = tid >> 4, d4 = tid & 15;
                for (int nd = node; nd < nrows; nd += 16) {
                    float4 m = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int hh = 0; hh < H; ++hh) {
                        const float4 y = lds128(stg_base + s * G::kStg + 1 * G::kStgT + nd * G::kRowB + hh * 256 + d4 * 16);
                        m.x += y.x; m.y += y.y; m.z += y.z; m.w += y.w;
                    }
                    const float inv = 1.f / (float)H;
                    const int64_t row = r0 + (int64_t)it * G::kNodes + nd;
                    *reinterpret_cast<float4*>(a.vbar + row * kDim + 4 * d4) = make_float4(m.x * inv, m.y * inv, m.z * inv, m.w * inv);
                }
            }
            if (it >= G::kNO) mbar_wait(&oempty[o], ((it / G::kNO) - 1) & 1);
            const uint32_t ob = ops_base + o * G::kOpStage;
#pragma unroll
            for (int i = 0; i < G::kChunksPerThread; ++i) {
                const int u = tid + 256 * i, node = u / G::kChunksPerRow, cc = u % G::kChunksPerRow;   // cc: 4-float column chunk
                const int head = cc >> 4, m = (cc & 15) * 4;
                const int blk = (H == 1) ? (node >> 4) : head;      // MN block of the UMMA
                const int kn = (H == 1) ? (node & 15) : node;        // K index (node inside the block tile)
                const uint32_t off = (uint32_t)(blk * G::kBlockTile + (kn >> 3) * 1024 + (kn & 7) * 128 +
                                                ((((m >> 3) ^ kn) & 7) << 4) + ((m >> 2) & 1) * 8);
                uint32_t hi[2], lo[2];
                if (!BWD) {
                    split4(x[i][0], hi, lo);
                    sts64(ob + 0 * G::kOp + off, hi[0], hi[1]);
                    sts64(ob + 1 * G::kOp + off, lo[0], lo[1]);
                    if (!a.gram) {
                        split4(x[i][1], hi, lo);
                        sts64(ob + 2 * G::kOp + off, hi[0], hi[1]);
                        sts64(ob + 3 * G::kOp + off, lo[0], lo[1]);
                    }
                    const float4 kk = x[i][0], vv = a.gram ? x[i][0] : x[i][1], qq = a.gram ? x[i][0] : x[i][2];
                    zacc[0] += kk.x; zacc[1] += kk.y; zacc[2] += kk.z; zacc[3] += kk.w;
                    uacc[0] += vv.x; uacc[1] += vv.y; uacc[2] += vv.z; uacc[3] += vv.w;
                    ssk = fmaf(kk.x, kk.x, ssk); ssk = fmaf(kk.y, kk.y, ssk); ssk = fmaf(kk.z, kk.z, ssk); ssk = fmaf(kk.w, kk.w, ssk);
                    ssq = fmaf(qq.x, qq.x, ssq); ssq = fmaf(qq.y, qq.y, ssq); ssq = fmaf(qq.z, qq.z, ssq); ssq = fmaf(qq.w, qq.w, ssq);
                } else {
                    // x[i][0] = q, x[i][1] = g, x[i][2] = out : 4 columns of (node, head); the 16 lanes of a
                    // (node, head) are consecutive -> xor-shuffle reductions inside the 16-lane group
                    const float4 qq = x[i][0], gg = x[i][1], oo = x[i][2];
                    const float4 zc4 = *reinterpret_cast<const float4*>(szc + cc * 4), u4 = *reinterpret_cast<const float4*>(su + cc * 4);
                    float qz = qq.x * zc4.x + qq.y * zc4.y + qq.z * zc4.z + qq.w * zc4.w;
                    float go = gg.x * oo.x + gg.y * oo.y + gg.z * oo.z + gg.w * oo.w;
                    float gu = gg.x * u4.x + gg.y * u4.y + gg.z * u4.z + gg.w * u4.w;
#pragma unroll
                    for (int sh_ = 1; sh_ < 16; sh_ <<= 1) {
                        qz += __shfl_xor_sync(0xffffffffu, qz, sh_);
                        go += __shfl_xor_sync(0xffffffffu, go, sh_);
                        gu += __shfl_xor_sync(0xffffffffu, gu, sh_);
                    }
                    const float inv = __frcp_rn(qz + a.n_total), dden = -go * inv;
                    const float4 dn = make_float4(gg.x * inv, gg.y * inv, gg.z * inv, gg.w * inv);
                    split4(qq, hi, lo);
                    sts64(ob + 0 * G::kOp + off, hi[0], hi[1]);
                    sts64(ob + 1 * G::kOp + off, lo[0], lo[1]);
                    split4(dn, hi, lo);
                    sts64(ob + 2 * G::kOp + off, hi[0], hi[1]);
                    sts64(ob + 3 * G::kOp + off, lo[0], lo[1]);
                    zacc[0] = fmaf(qq.x, dden, zacc[0]); zacc[1] = fmaf(qq.y, dden, zacc[1]);
                    zacc[2] = fmaf(qq.z, dden, zacc[2]); zacc[3] = fmaf(qq.w, dden, zacc[3]);
                    uacc[0] += dn.x; uacc[1] += dn.y; uacc[2] += dn.z; uacc[3] += dn.w;
                    if ((cc & 15) == 0 && node < nrows) {
                        ssq += go - inv * gu + dden * qz;           // t_q contribution of this (node, head)
                        const int64_t row = r0 + (int64_t)it * G::kNodes + node;
                        *reinterpret_cast<float2*>(a.rowscal + (row * H + head) * 2) = make_float2(inv, dden);
                    }
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) { mbar_arrive(&ofull[o]); mbar_arrive(&sempty[s]); }
        }
    } else if (warp == 8) {
        if (lane == 0) {
            // ===== TMA issuer: the stage's rows of K, V, Q are contiguous in HBM: three bulk copies per stage
            const uint32_t stg_base = smem_u32(stg);
            const uint64_t pol_first = policy_evict_first_(), pol_last = policy_evict_last();
            for (int it = 0; it < iters; ++it) {
                const int s = it % G::kNSG;
                if (it >= G::kNSG) mbar_wait(&sempty[s], ((it / G::kNSG) - 1) & 1);
                const int64_t row = r0 + (int64_t)it * G::kNodes;
                const uint32_t bytes = (uint32_t)(min((int64_t)G::kNodes, r1 - row) * G::kRowB);
                if (!BWD && a.gram) {   // K = V = Q = the layer input: one copy; pass 2 reads it again
                    mbar_expect_tx(&sfull[s], bytes);
                    tma_load_1d_hint(stg_base + s * G::kStg + 0 * G::kStgT, a.k + row * G::kRowF, bytes, &sfull[s], pol_last);
                    continue;
                }
                mbar_expect_tx(&sfull[s], 3 * bytes);
                if (a.l2_hints) {     // K, V are dead after this pass; Q is read again by pass 2
                    tma_load_1d_hint(stg_base + s * G::kStg + 0 * G::kStgT, a.k + row * G::kRowF, bytes, &sfull[s], pol_first);
                    tma_load_1d_hint(stg_base + s * G::kStg + 1 * G::kStgT, a.v + row * G::kRowF, bytes, &sfull[s], pol_first);
                    tma_load_1d_hint(stg_base + s * G::kStg + 2 * G::kStgT, a.q + row * G::kRowF, bytes, &sfull[s], pol_last);
                } else {
                    tma_load_1d(stg_base + s * G::kStg + 0 * G::kStgT, a.k + row * G::kRowF, bytes, &sfull[s]);
                    tma_load_1d(stg_base + s * G::kStg + 1 * G::kStgT, a.v + row * G::kRowF, bytes, &sfull[s]);
                    tma_load_1d(stg_base + s * G::kStg + 2 * G::kStgT, a.q + row * G::kRowF, bytes, &sfull[s]);
                }
            }
        }
    } else if (lane == 0) {
        // ===== MMA issuer: D_p[128 x 128] += A^T B over 16 K-steps-worth of nodes; MN-major operands
        const uint32_t idesc = make_idesc(128, 128, 1, 1);
        const uint32_t lbo = G::kBlockTile, sbo = 1024;
        const uint32_t ops_base = smem_u32(ops);
        for (int it = 0; it < iters; ++it) {
            const int o = it % G::kNO;
            mbar_wait(&ofull[o], (it / G::kNO) & 1);
            tc_fence_after();
            const uint32_t sb = ops_base + o * G::kOpStage;
#pragma unroll
            for (int p = 0; p < G::kPairs; ++p) {
                const uint32_t ho = p * 2 * G::kBlockTile;
                const uint64_t khi = make_desc(sb + 0 * G::kOp + ho, lbo, sbo), klo = make_desc(sb + 1 * G::kOp + ho, lbo, sbo);
                const bool same = !BWD && a.gram;      // X^T X: the K operand on both sides
                const uint64_t vhi = same ? khi : make_desc(sb + 2 * G::kOp + ho, lbo, sbo), vlo = same ? klo : make_desc(sb + 3 * G::kOp + ho, lbo, sbo);
                umma(tmem + p * 128, khi, vhi, idesc, it > 0 ? 1u : 0u);
                umma(tmem + p * 128, khi, vlo, idesc, 1u);
                umma(tmem + p * 128, klo, vhi, idesc, 1u);
            }
            umma_commit(&oempty[o]);
        }
        if (iters > 0) umma_commit(&done); else mbar_arrive(&done);
    }

    // ===== tail: per-CTA record in the partials layout [S | z | u | sq | sk], then the cross-CTA sum fused in:
    // every CTA publishes its record (flag = epoch), waits for all flags (cooperative launch: all CTAs are resident),
    // gathers "its" column slices of all records with TMA and sums them in a fixed order (fp64) -> partials
    // (deterministic, no float atomics).  S / z entries are also emitted as the pass-2 operand image (bf16 hi/lo, swizzled).
    __syncwarp();
    if (warp == 0) DIF_STAMP(dbg, 3);
    mbar_wait(&done, 0);
    tc_fence_after();
    DIF_STAMP(dbg, 4);
    ssk = warp_sum(ssk);
    ssq = warp_sum(ssq);
    if (lane == 0 && warp < 8) { part[warp] = ssk; part[8 + warp] = ssq; }
    float* red = reinterpret_cast<float*>(ops);         // all MMAs have completed: operand memory is free
    if (warp < 8) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { red[tid * 4 + i] = zacc[i]; red[1024 + tid * 4 + i] = uacc[i]; }
    }
    __syncthreads();
    float* rec = a.ws + (int64_t)blockIdx.x * a.ws_len;
    if (tid < G::kRowF) {
        // column tid = chunk (tid >> 2) element (tid & 3); the threads t with t mod 16H == chunk hold its partial sums
        float z = 0.f, u = 0.f;
        for (int t = tid >> 2; t < 256; t += G::kChunksPerRow) { z += red[t * 4 + (tid & 3)]; u += red[1024 + t * 4 + (tid & 3)]; }
        rec[G::offZ + tid] = z;
        rec[G::offU + tid] = u;
    }
    if (tid == 0) {
        float sk = 0.f, sq = 0.f;
        for (int w = 0; w < 8; ++w) { sk += part[w]; sq += part[8 + w]; }
        rec[G::offSq] = sq;                  // fwd: sum q^2 ; bwd: t_q
        rec[G::offSq + 1] = BWD ? 0.f : sk;  // fwd: sum k^2 ; bwd: t_k is filled in later (needs the reduced dS)
        for (int64_t i = G::kP; i < a.ws_len; ++i) rec[i] = 0.f;
    }
    __syncthreads();                                   // `red` is re-used below (H == 1)
    {
        // D_p rows 0-63 x cols 0-63 = block 2p, rows 64-127 x cols 64-127 = block 2p+1.  Warp w reads TMEM lanes
        // 32(w%4)..+31 (its quadrant); warps 0-3 take pair 0, warps 4-7 pair 1 (H = 4 only).
        const int wq = warp & 3, p = warp >> 2;
        const int hp = wq >> 1, m = (wq * 32 + lane) & 63;
        const bool active = warp < 4 * G::kPairs;
        uint32_t r[2][32];
        if (active) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                if (iters > 0) {
                    tmem_ld32(tmem + ((uint32_t)(wq * 32) << 16) + p * 128 + hp * 64 + c * 32, r[c]);
                    tmem_ld_wait32(r[c]);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[c][j] = 0u;
                }
            }
        }
        if (H == 1) {
            // the two diagonal blocks are the two node halves of every stage: S = block 0 + block 1
            if (active && hp == 1) {
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int j = 0; j < 32; ++j) red[m * 65 + c * 32 + j] = __uint_as_float(r[c][j]);
            }
            __syncthreads();
            if (active && hp == 0) {
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[c][j] = __float_as_uint(__uint_as_float(r[c][j]) + red[m * 65 + c * 32 + j]);
            }
        }
        if (active && (H != 1 || hp == 0)) {
            const int blk = (H == 1) ? 0 : 2 * p + hp;
            float* dst = rec + ((int64_t)blk * kDim + m) * kDim;
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
                for (int j = 0; j < 32; j += 8)
                    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                                 :: "l"(dst + c * 32 + j), "r"(r[c][j]), "r"(r[c][j + 1]), "r"(r[c][j + 2]), "r"(r[c][j + 3]),
                                    "r"(r[c][j + 4]), "r"(r[c][j + 5]), "r"(r[c][j + 6]), "r"(r[c][j + 7]) : "memory");
        }
    }
    // ---- publish the record
    __threadfence();
    __syncthreads();
    DIF_STAMP(dbg, 5);
    const int grid = gridDim.x;
    // epoch = host value + device-side generation word (flags[grid], any initial value; CTA 0 bumps it once every CTA
    // has published, i.e. after every CTA has read it): a CUDA-graph replay repeats the host value, never the epoch
    const unsigned long long gen = *reinterpret_cast<volatile unsigned long long*>(a.flags + grid);
    const unsigned long long epoch = a.epoch + gen * 0x9E3779B97F4A7C15ull;
    if (tid == 0) asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(a.flags + blockIdx.x), "l"(epoch) : "memory");
    // ---- column slices of the record: kSlices fixed slices of `chunk` floats (multiples of 16 B), slice sl is owned by
    //      CTA sl % grid -- the partition does not depend on this rank's grid, so slices line up across ranks
    const int chunk = (int)((((a.ws_len + kSlices - 1) / kSlices) + 3) & ~(int64_t)3);
    float* sbuf = reinterpret_cast<float*>(stg);        // [grid][chunk] fp32, the staging ring is idle now
    const ShardArgs& sh = a.sh;
    const bool sharded = sh.world > 1;
    const int xslot = (int)(sh.seq & 1);
    if (sharded && blockIdx.x == 0 && tid == 0) comm_check_status(sh);
    bool waited = false;
    uint32_t tail_phase = 0;
    for (int sl = blockIdx.x; sl < kSlices; sl += grid) {
        const int64_t j0 = (int64_t)sl * chunk;
        const int slice = (int)max((int64_t)0, min(a.ws_len, j0 + chunk) - j0);
        if (slice <= 0) break;
        if (!waited) {
            for (int r = tid; r < grid; r += kThreadsT) {
                unsigned long long f;
                do {
                    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(f) : "l"(a.flags + r) : "memory");
                    if (f != epoch) __nanosleep(64);
                } while (f != epoch);
            }
            if (blockIdx.x == 0) {
                __syncthreads();
                if (tid == 0) *reinterpret_cast<volatile unsigned long long*>(a.flags + grid) = gen + 1;
            }
            asm volatile("fence.proxy.async;" ::: "memory");   // acquired (generic proxy) before the bulk (async proxy) reads
            waited = true;
        }
        __syncthreads();                                  // also: the previous slice's readers of sbuf are done
        if (tid == 0) mbar_expect_tx(&tail_bar, (uint32_t)grid * (uint32_t)slice * 4u);
        __syncthreads();
        for (int r = tid; r < grid; r += kThreadsT)
            tma_load_1d(smem_u32(sbuf) + (uint32_t)r * chunk * 4, a.ws + (int64_t)r * a.ws_len + j0, (uint32_t)slice * 4u, &tail_bar);
        mbar_wait(&tail_bar, tail_phase);
        tail_phase ^= 1;
        const int t = tid;                                // chunk <= kThreadsT (checked on the host)
        const int64_t j = j0 + t;
        const bool live = t < slice && j < G::kP;
        float local = 0.f;
        if (live) {
            // four independent chains (records r = 4i + k), combined in a fixed order: deterministic, 4x shorter latency
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            int r = 0;
            for (; r + 3 < grid; r += 4) {
                a0 += (double)sbuf[(r + 0) * chunk + t];
                a1 += (double)sbuf[(r + 1) * chunk + t];
                a2 += (double)sbuf[(r + 2) * chunk + t];
                a3 += (double)sbuf[(r + 3) * chunk + t];
            }
            for (; r < grid; ++r) a0 += (double)sbuf[r * chunk + t];
            local = (float)((a0 + a1) + (a2 + a3));
        }
        float sum = local;
        if (sharded) {
            // ---- cross-GPU: the same kernel finishes the all-reduce over NVLink, slice by slice, LL push protocol
            // (common.cuh): element j of the local slice goes straight into every peer's LL region as one 64-bit word
            // {call number | fp32}; then the peers' words are polled in the LOCAL region and added in rank order
            // (bit-identical on all ranks).  One NVLink traversal on the critical path, no fence, no flag round trip.
            const uint32_t tag = (uint32_t)sh.seq;
            if (live) {
                for (int p = 1; p < sh.world; ++p) {          // start at the next rank: spreads the targets over the switch
                    int r = sh.rank + p;
                    if (r >= sh.world) r -= sh.world;
                    comm_ll_send(comm_ll_ptr(sh.bufs[r], sh.lenpad, xslot, sh.rank) + j, local, tag);
                }
                sum = comm_ll_sum(sh, xslot, j, tag, local);
            }
        }
        if (live) {
            a.partials[j] = sum;
            if (!BWD && a.prepared != nullptr && j < G::offU) {
                // B operand image of pass 2 (un-scaled; pass 2 applies c = 1/(|Q||K|) in its epilogue):
                // S[h][m][d] -> row n = d, k = m of head h ; z[h][m] -> row 64
                int h, n, m;
                if (j < G::offZ) { h = (int)(j >> 12); m = (int)(j >> 6) & 63; n = (int)j & 63; }
                else { h = (int)(j - G::offZ) >> 6; m = (int)(j - G::offZ) & 63; n = kDim; }
                const __nv_bfloat16 hi = __float2bfloat16_rn(sum);
                const __nv_bfloat16 lo = __float2bfloat16_rn(sum - __bfloat162float(hi));
                uint8_t* img = a.prepared + (size_t)h * 2 * kBOp + sw128(n, m >> 3) + (m & 7) * 2;
                *reinterpret_cast<__nv_bfloat16*>(img) = hi;
                *reinterpret_cast<__nv_bfloat16*>(img + kBOp) = lo;
            }
        }
    }
    if (!BWD && a.prepared != nullptr && blockIdx.x == grid - 1) {
        // rows 65..79 of every (head, hi|lo) tile are zero padding (N = 80 of the pass-2 UMMA)
        for (int i = tid; i < H * 2 * 15 * 8; i += kThreadsT) {
            const int c = i & 7, rr = (i >> 3) % 15 + 65, t = i / (8 * 15);
            *reinterpret_cast<uint4*>(a.prepared + (size_t)t * kBOp + sw128(rr, c)) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    tc_fence_before();
    __syncthreads();
    DIF_STAMP(dbg, 6);
    if (warp == 9) tmem_dealloc(tmem, G::kTmemCols1);
}

// ------------------------------------------------------------------------------------------
// pass 2
// ------------------------------------------------------------------------------------------
struct ApplyTcArgs {
    // A operand rows: element (row, head h, column c) at q[row * q_ld + h * q_hs + c].  Plain [N,H,64] queries: q_ld = 64 H, q_hs = 64.
    // Projection folded into the operands (dif_simple_apply_projected): q = the layer input x [N,64], q_ld = 64, q_hs = 0 (every head
    // re-reads the same x tile, from L2) and `nvec` holds one denominator constant per head.
    int64_t q_ld;
    int q_hs;
    const float* nvec;
    const float* q;
    const float* partials;
    float n_total;
    int64_t N;
    float* out;
    int pf_tiles;            // L2 prefetch distance in tiles (0 = off)
    int store_hint;          // 1: TMA stores carry an L2 evict_first policy (the output is not re-read)
    uint64_t* dbg;           // optional timeline buffer
    const uint8_t* prepared; // optional B operand image written by the fused pass-1 tail (un-scaled S|z, bf16 hi/lo, swizzled)
    dif_epilogue_t ep;
};

// SHARED: the H heads of a tile use ONE A operand (q_hs == 0: the projected form, A = the layer input x): a stage is a tile, loaded and
// split once, and the issuer runs the H head MMAs (N = 80 each, their own accumulator slots) off it.
template <int H, bool SHARED = false>
__global__ void __launch_bounds__(kThreadsTC, 1) apply_tc_kernel(const __grid_constant__ ApplyTcArgs p, const __grid_constant__ CUtensorMap out_map) {
    using G = Geo<H>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* Bop = base;                                             // [h][hi|lo][80 rows][128 B]
    uint8_t* stages = base + G::kBBytes;
    uint8_t* ostage = stages + kNS2 * kStage2;                       // [4 warps][2 boxes][32 rows][128 B], 1024-aligned
    float* us = reinterpret_cast<float*>(ostage + kOutStage);        // [H][64]
    __shared__ uint64_t full[kNS2], empty[kNS2], tfull[kNAcc], tempty[kNAcc], bbar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t ntiles = (p.N + kTile2 - 1) / kTile2;
    const int my_tiles = blockIdx.x < ntiles ? (int)((ntiles - 1 - blockIdx.x) / gridDim.x + 1) : 0;
    const int nsc = my_tiles * H;                       // (tile, head) units of this CTA
    const int nst = SHARED ? my_tiles : nsc;            // A-operand stages
    auto tile_of = [&](int sc) -> int64_t { return blockIdx.x + (int64_t)(sc / H) * gridDim.x; };

    DIF_STAMP(p.dbg, 0);
    if (tid == 32 && my_tiles > 0) {
        // have the first tiles of Q on their way to L2 while the prologue runs
        for (int i = 0; i < 2 && i < my_tiles; ++i) {
            const int64_t prow = tile_of(H * i) * kTile2;
            const int64_t nrows = min((int64_t)kTile2, p.N - prow);
            for (int64_t r = 0; r < nrows; r += 16)
                prefetch_l2(p.q + (prow + r) * p.q_ld, (uint32_t)(min((int64_t)16, nrows - r) * p.q_ld * 4));
        }
    }
    if (tid == 0) {
        for (int s = 0; s < kNS2; ++s) { mbar_init(&full[s], 8); mbar_init(&empty[s], 1); }
        for (int s = 0; s < kNAcc; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 4); }
        mbar_init(&bbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (p.prepared != nullptr) {
            // the B operands were prepared by pass 1: one TMA fetch instead of a transposing prologue
            mbar_expect_tx(&bbar, (uint32_t)G::kBBytes);
            for (int i = 0; i < H * 2; ++i)
                tma_load_1d(smem_u32(Bop) + i * kBOp, p.prepared + (size_t)i * kBOp, (uint32_t)kBOp, &bbar);
        }
    }
    if (warp == 12) tmem_alloc(&tmem_slot, 512);

    // ---- B operands: row n < 64: S[h][:, n] ; row 64: z[h] ; rows 65..79: 0   (K-major SW128, hi/lo split)
    const float c = 1.f / (sqrtf(p.partials[G::offSq]) * sqrtf(p.partials[G::offSq + 1]));
    const float cscale = p.prepared != nullptr ? c : 1.f;   // prepared operands are un-scaled: the epilogue applies c
    if (p.prepared == nullptr) {
        // fallback (partials were edited / all-reduced outside): build the operands here, pre-scaled by c.
        // All loads of a thread's tasks are issued before the first use: two L2 round trips, not 50.
        constexpr int kTasks = H * 8 * kBN, kPer = (kTasks + kThreadsTC - 1) / kThreadsTC;
        float x[kPer][8];
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int task = tid + u * kThreadsTC;
            const int n = task % kBN, hc = task / kBN, ch = hc & 7, h = hc >> 3;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int m = ch * 8 + i;
                x[u][i] = 0.f;
                if (task < kTasks) {
                    if (n < kDim) x[u][i] = __ldg(p.partials + ((int64_t)h * kDim + m) * kDim + n);
                    else if (n == kDim) x[u][i] = __ldg(p.partials + G::offZ + h * kDim + m);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int task = tid + u * kThreadsTC;
            if (task < kTasks) {
                const int n = task % kBN, hc = task / kBN, ch = hc & 7, h = hc >> 3;
#pragma unroll
                for (int i = 0; i < 8; ++i) x[u][i] *= c;
                uint4 hi, lo;
                split8(x[u], hi, lo);
                const uint32_t off = (uint32_t)(h * 2 * kBOp) + sw128(n, ch);
                sts128(smem_u32(Bop) + off, hi);
                sts128(smem_u32(Bop) + kBOp + off, lo);
            }
        }
    }
    for (int i = tid; i < H * kDim; i += kThreadsTC) us[i] = p.partials[G::offU + i];
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    DIF_STAMP(p.dbg, 1);

    if (warp < 8) {
        // ===== Q producers: stage = (tile, head): 128 rows x 256 B; task t -> row t>>3, chunk t&7.
        // Whole-stage double buffer: buf[0] = current, buf[1] = next (its loads are in flight while buf[0] is converted).
        float buf[2][4][8];
        auto issue = [&](int st, int j, float (&dst)[8]) {
            if (st >= nst) return;
            const int64_t tile = tile_of(SHARED ? st * H : st);
            const int t = tid + 256 * j;
            const int64_t row = tile * kTile2 + (t >> 3);
            if (row < p.N) {
                if (!SHARED && p.q_hs != 0) ldg256_stream(p.q + row * p.q_ld + (st % H) * p.q_hs + (t & 7) * 8, dst);
                else ldg256_keep(p.q + row * p.q_ld + (t & 7) * 8, dst);         // shared by the heads: let it stay in L2
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[i] = 0.f;
            }
        };
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(0, j, buf[0][j]);
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(1, j, buf[1][j]);
        const uint32_t stage_base = smem_u32(stages);
        for (int st = 0; st < nst; ++st) {
            const int s = st % kNS2;
            if (st >= kNS2) mbar_wait(&empty[s], ((st / kNS2) - 1) & 1);
            const uint32_t sb = stage_base + s * kStage2;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = tid + 256 * j;
                uint4 hi, lo;
                split8(buf[0][j], hi, lo);
                const uint32_t off = sw128(t >> 3, t & 7);
                sts128(sb + off, hi);
                sts128(sb + kQOp + off, lo);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
            if (st == 0) DIF_STAMP(p.dbg, 2);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int i = 0; i < 8; ++i) buf[0][j][i] = buf[1][j][i];
                issue(st + 2, j, buf[1][j]);
            }
        }
    } else if (warp < 12) {
        // ===== epilogue: thread = one row of the tile; accumulator lane = 32*(warp%4) + lane.  Results leave through TMA:
        // each lane writes its row into a 128B-swizzled staging box (conflict-free st.shared), one lane issues
        // cp.async.bulk.tensor stores (rows beyond N are clipped by the tensor map).  No scattered st.global on the LSU.
        const int ew = warp - 8;
        const uint32_t obox = smem_u32(ostage) + ew * 2 * kOutBox;
        const uint64_t pol = policy_evict_first();
        for (int sc = 0; sc < nsc; ++sc) {
            const int64_t tile = tile_of(sc);
            const int h = sc % H, slot = sc % kNAcc;
            mbar_wait(&tfull[slot], (sc / kNAcc) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(ew * 32) << 16) + slot * kAccCols;
            uint32_t qz_bits = tmem_ld1(taddr + kDim);            // column 64 = q . z
            tmem_ld_wait1(qz_bits);
            const float inv_den = 1.f / (fmaf(__uint_as_float(qz_bits), cscale, p.nvec != nullptr ? __ldg(p.nvec + h) : p.n_total));   // one division per (row, head)
            if (lane == 0) tma_wait_read0();      // staging is about to be rewritten: previous TMA reads must be done
            __syncwarp();
#pragma unroll
            for (int c0 = 0; c0 < kDim; c0 += 32) {
                uint32_t r[32];
                tmem_ld32(taddr + c0, r);
                tmem_ld_wait32(r);
                if (c0 == 32) {          // everything of this slot is in registers: hand the accumulator back
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tempty[slot]);
                }
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 u4 = *reinterpret_cast<const float4*>(us + h * kDim + c0 + j);
                    float4 o;
                    o.x = fmaf(__uint_as_float(r[j]), cscale, u4.x) * inv_den;
                    o.y = fmaf(__uint_as_float(r[j + 1]), cscale, u4.y) * inv_den;
                    o.z = fmaf(__uint_as_float(r[j + 2]), cscale, u4.z) * inv_den;
                    o.w = fmaf(__uint_as_float(r[j + 3]), cscale, u4.w) * inv_den;
                    sts128(obox + (c0 >> 5) * kOutBox + sw128(lane, j >> 2),
                           make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(o.w)));
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                const int col = h * kDim;
                const int row0 = (int)(tile * kTile2) + ew * 32;
                if (p.store_hint) {
                    tma_store_2d_hint(&out_map, obox, col, row0, pol);
                    tma_store_2d_hint(&out_map, obox + kOutBox, col + 32, row0, pol);
                } else {
                    tma_store_2d(&out_map, obox, col, row0);
                    tma_store_2d(&out_map, obox + kOutBox, col + 32, row0);
                }
                tma_commit();
            }
            if (sc == H - 1 && ew == 0 && lane == 0) DIF_STAMP_ANY(p.dbg, 6);
        }
        if (ew == 0 && lane == 0) DIF_STAMP_ANY(p.dbg, 8);
        if (lane == 0) tma_wait_all0();      // stores must have landed before the CTA exits
        if (ew == 0 && lane == 0) DIF_STAMP_ANY(p.dbg, 9);
    } else if (lane == 0) {
        // ===== MMA issuer: per (tile, head): 4 K-steps x (hi*hi + lo*hi + hi*lo), M=128 N=80 K=16
        const uint32_t idesc = make_idesc(kTile2, kBN, 0, 0);
        const uint32_t stage_base = smem_u32(stages), b_base = smem_u32(Bop);
        if (p.prepared != nullptr) mbar_wait(&bbar, 0);
        for (int st = 0; st < nst; ++st) {
            const int s = st % kNS2;
            const int sc0 = SHARED ? st * H : st;
            if (p.pf_tiles > 0 && sc0 % H == 0 && sc0 + H * p.pf_tiles < nsc) {
                const int64_t prow = tile_of(sc0 + H * p.pf_tiles) * kTile2;
                const int64_t nrows = min((int64_t)kTile2, p.N - prow);
                for (int64_t r = 0; r < nrows; r += 16)
                    prefetch_l2(p.q + (prow + r) * p.q_ld, (uint32_t)(min((int64_t)16, nrows - r) * p.q_ld * 4));
            }
            bool have_a = false;
#pragma unroll
            for (int hh = 0; hh < (SHARED ? H : 1); ++hh) {
                const int sc = sc0 + hh, slot = sc % kNAcc, h = sc % H;
                if (sc >= kNAcc) mbar_wait(&tempty[slot], ((sc / kNAcc) - 1) & 1);
                if (!have_a) { mbar_wait(&full[s], (st / kNS2) & 1); have_a = true; }
                tc_fence_after();
                const uint32_t sb = stage_base + s * kStage2, bb = b_base + h * 2 * kBOp;
                const uint32_t d = tmem + slot * kAccCols;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint64_t qhi = make_desc(sb + ks * 32, kKmajLBO, kKmajSBO), qlo = make_desc(sb + kQOp + ks * 32, kKmajLBO, kKmajSBO);
                    const uint64_t bhi = make_desc(bb + ks * 32, kKmajLBO, kKmajSBO), blo = make_desc(bb + kBOp + ks * 32, kKmajLBO, kKmajSBO);
                    umma(d, qhi, bhi, idesc, ks > 0 ? 1u : 0u);
                    umma(d, qlo, bhi, idesc, 1u);
                    umma(d, qhi, blo, idesc, 1u);
                }
                if (hh == (SHARED ? H : 1) - 1) umma_commit(&empty[s]);
                umma_commit(&tfull[slot]);
            }
        }
        DIF_STAMP_ANY(p.dbg, 7);
    }
    __syncwarp();
    if (warp == 0) DIF_STAMP(p.dbg, 3);
    tc_fence_before();
    __syncthreads();
    DIF_STAMP(p.dbg, 5);
    if (warp == 12) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------
// Pass 2 with the layer epilogue (mode 1: head mean, gcn / x_0 / residual addends, LayerNorm, ReLU; difformer.py:129-140, 200-203),
// 17 warps.  Same producers, stage ring, B operands and MMA issue as apply_tc_kernel; what differs is the epilogue, which was the
// limiter of apply_tc_kernel<1,...> (one thread per output row: ~1400 dependent instructions per tile on one warp per scheduler,
// 8.5 us per tile): here TWO threads share a row -- warps 8-11 take columns 0-31 of every head, warps 12-15 columns 32-63 (a warp
// may read the TMEM lanes 32 (warp % 4) .. +31, so the pair (w, w + 4) sees the same rows) -- and the LayerNorm statistics cross the
// pair through shared memory and a 64-thread named barrier.  Half the work per thread, two epilogue warps per scheduler.
// ------------------------------------------------------------------------------------------
constexpr int kLayerWarps = 17, kLayerThreads = kLayerWarps * 32;

template <int H, bool SHARED>
__global__ void __launch_bounds__(kLayerThreads, 1) layer_tc_kernel(const __grid_constant__ ApplyTcArgs p, const __grid_constant__ CUtensorMap out_map) {
    using G = Geo<H>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* Bop = base;                                             // [h][hi|lo][80 rows][128 B]
    uint8_t* stages = base + G::kBBytes;
    uint8_t* ostage = stages + kNS2 * kStage2;                       // [8 warps][32 rows][128 B], 1024-aligned
    float* us = reinterpret_cast<float*>(ostage + kOutStage);        // [H][64]
    __shared__ uint64_t full[kNS2], empty[kNS2], tfull[kNAcc], tempty[kNAcc], bbar;
    __shared__ uint32_t tmem_slot;
    __shared__ float ln_sum[2][kTile2], ln_var[2][kTile2];           // LayerNorm partial statistics of the two column halves
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t ntiles = (p.N + kTile2 - 1) / kTile2;
    const int my_tiles = blockIdx.x < ntiles ? (int)((ntiles - 1 - blockIdx.x) / gridDim.x + 1) : 0;
    const int nsc = my_tiles * H;                       // (tile, head) units of this CTA
    const int nst = SHARED ? my_tiles : nsc;            // A-operand stages
    auto tile_of = [&](int sc) -> int64_t { return blockIdx.x + (int64_t)(sc / H) * gridDim.x; };

    DIF_STAMP(p.dbg, 0);
    if (tid == 0) {
        for (int s = 0; s < kNS2; ++s) { mbar_init(&full[s], 8); mbar_init(&empty[s], 1); }
        for (int s = 0; s < kNAcc; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 8); }
        mbar_init(&bbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (p.prepared != nullptr) {
            mbar_expect_tx(&bbar, (uint32_t)G::kBBytes);
            for (int i = 0; i < H * 2; ++i)
                tma_load_1d(smem_u32(Bop) + i * kBOp, p.prepared + (size_t)i * kBOp, (uint32_t)kBOp, &bbar);
        }
    }
    if (warp == 16) tmem_alloc(&tmem_slot, 512);

    // ---- B operands (see apply_tc_kernel): row n < 64: S[h][:, n]; row 64: z[h]; rows 65..79: 0   (K-major SW128, hi/lo split)
    const float c = 1.f / (sqrtf(p.partials[G::offSq]) * sqrtf(p.partials[G::offSq + 1]));
    const float cscale = p.prepared != nullptr ? c : 1.f;
    if (p.prepared == nullptr) {
        constexpr int kTasks = H * 8 * kBN, kPer = (kTasks + kLayerThreads - 1) / kLayerThreads;
        float x[kPer][8];
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int task = tid + u * kLayerThreads;
            const int n = task % kBN, hc = task / kBN, ch = hc & 7, h = hc >> 3;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int m = ch * 8 + i;
                x[u][i] = 0.f;
                if (task < kTasks) {
                    if (n < kDim) x[u][i] = __ldg(p.partials + ((int64_t)h * kDim + m) * kDim + n);
                    else if (n == kDim) x[u][i] = __ldg(p.partials + G::offZ + h * kDim + m);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int task = tid + u * kLayerThreads;
            if (task < kTasks) {
                const int n = task % kBN, hc = task / kBN, ch = hc & 7, h = hc >> 3;
#pragma unroll
                for (int i = 0; i < 8; ++i) x[u][i] *= c;
                uint4 hi, lo;
                split8(x[u], hi, lo);
                const uint32_t off = (uint32_t)(h * 2 * kBOp) + sw128(n, ch);
                sts128(smem_u32(Bop) + off, hi);
                sts128(smem_u32(Bop) + kBOp + off, lo);
            }
        }
    }
    for (int i = tid; i < H * kDim; i += kLayerThreads) us[i] = p.partials[G::offU + i];
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    DIF_STAMP(p.dbg, 1);

    if (warp < 8) {
        // ===== A producers (see apply_tc_kernel): stage = tile (SHARED) or (tile, head)
        float buf[2][4][8];
        auto issue = [&](int st, int j, float (&dst)[8]) {
            if (st >= nst) return;
            const int64_t tile = tile_of(SHARED ? st * H : st);
            const int t = tid + 256 * j;
            const int64_t row = tile * kTile2 + (t >> 3);
            if (row < p.N) {
                if (!SHARED && p.q_hs != 0) ldg256_stream(p.q + row * p.q_ld + (st % H) * p.q_hs + (t & 7) * 8, dst);
                else ldg256_keep(p.q + row * p.q_ld + (t & 7) * 8, dst);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[i] = 0.f;
            }
        };
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(0, j, buf[0][j]);
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(1, j, buf[1][j]);
        const uint32_t stage_base = smem_u32(stages);
        for (int st = 0; st < nst; ++st) {
            const int s = st % kNS2;
            if (st >= kNS2) mbar_wait(&empty[s], ((st / kNS2) - 1) & 1);
            const uint32_t sb = stage_base + s * kStage2;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = tid + 256 * j;
                uint4 hi, lo;
                split8(buf[0][j], hi, lo);
                const uint32_t off = sw128(t >> 3, t & 7);
                sts128(sb + off, hi);
                sts128(sb + kQOp + off, lo);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
            if (st == 0) DIF_STAMP(p.dbg, 2);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int i = 0; i < 8; ++i) buf[0][j][i] = buf[1][j][i];
                issue(st + 2, j, buf[1][j]);
            }
        }
    } else if (warp < 16) {
        // ===== epilogue: thread = (row, column half).  TMEM lane = 32 * quad + lane, columns 32 * half .. +31 of each head
        const int ew = warp - 8, quad = ew & 3, half = ew >> 2;
        const uint32_t obox = smem_u32(ostage) + ew * kOutBox;
        const uint64_t pol = policy_evict_first();
        const int lrow = quad * 32 + lane;              // row inside the tile
        float hs[32];
        int inflight = -1, pending = 0;                 // addend whose copy is in flight / next addend to fetch
        int64_t row = 0;
        auto cp_issue = [&](int a) {
            const float* src = p.ep.add[a] + row * kDim + 32 * half;
#pragma unroll
            for (int j = 0; j < 8; ++j) cp_async16(obox + sw128(lane, j), src + 4 * j);
            cp_async_commit();
        };
        auto cp_fold = [&]() {                          // wait for the addend in flight, add it, start the next one
            cp_async_wait_all();
            const float s = p.ep.add_scale[inflight];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 x = lds128(obox + sw128(lane, j));
                hs[4 * j] = fmaf(s, x.x, hs[4 * j]); hs[4 * j + 1] = fmaf(s, x.y, hs[4 * j + 1]);
                hs[4 * j + 2] = fmaf(s, x.z, hs[4 * j + 2]); hs[4 * j + 3] = fmaf(s, x.w, hs[4 * j + 3]);
            }
            inflight = -1;
            if (pending < p.ep.n_add) { cp_issue(pending); inflight = pending++; }
        };
        for (int sc = 0; sc < nsc; ++sc) {
            const int64_t tile = tile_of(sc);
            const int h = sc % H, slot = sc % kNAcc;
            row = tile * kTile2 + lrow;
            const bool ok = row < p.N;
            if (h == 0) {
                // Addends (gcn term, x_0, residual): this thread's 128-byte piece of each goes global -> its row of the warp's staging
                // box by cp.async (no registers in flight) and is folded in after the next head's arithmetic, one addend behind one
                // head; the rows of the CTA's next tile are pulled into L2 meanwhile.  The box is free once the previous tile's TMA
                // store has read it.
#pragma unroll
                for (int i = 0; i < 32; ++i) hs[i] = 0.f;
                if (lane == 0) tma_wait_read0();
                __syncwarp();
                inflight = -1;
                pending = 0;
                if (ok && p.ep.n_add > 0) { cp_issue(0); inflight = 0; pending = 1; }
                const int64_t nrow = row + (int64_t)gridDim.x * kTile2;
                if (nrow < p.N)
                    for (int a = 0; a < p.ep.n_add; ++a) prefetch_l2_line(p.ep.add[a] + nrow * kDim + 32 * half);
            }
            mbar_wait(&tfull[slot], (sc / kNAcc) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(quad * 32) << 16) + slot * kAccCols;
            uint32_t qz_bits = tmem_ld1(taddr + kDim);            // column 64 = q . z
            uint32_t r[32];
            tmem_ld32(taddr + 32 * half, r);
            tmem_ld_wait32(r);
            tmem_ld_wait1(qz_bits);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[slot]);             // everything of this slot is in registers
            const float inv_den = p.ep.attn_scale / fmaf(__uint_as_float(qz_bits), cscale, p.nvec != nullptr ? __ldg(p.nvec + h) : p.n_total);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 u4 = *reinterpret_cast<const float4*>(us + h * kDim + 32 * half + j);
                hs[j] = fmaf(fmaf(__uint_as_float(r[j]), cscale, u4.x), inv_den, hs[j]);
                hs[j + 1] = fmaf(fmaf(__uint_as_float(r[j + 1]), cscale, u4.y), inv_den, hs[j + 1]);
                hs[j + 2] = fmaf(fmaf(__uint_as_float(r[j + 2]), cscale, u4.z), inv_den, hs[j + 2]);
                hs[j + 3] = fmaf(fmaf(__uint_as_float(r[j + 3]), cscale, u4.w), inv_den, hs[j + 3]);
            }
            if (inflight >= 0) cp_fold();
            if (h != H - 1) continue;
            while (inflight >= 0) cp_fold();             // more addends than heads
            if (p.ep.gcn_rowptr != nullptr && ok) {
                // gcn_conv term gathered here (optional, see apply_tc_kernel): this thread's half of the neighbour rows
                const int beg = __ldg(p.ep.gcn_rowptr + row), end = __ldg(p.ep.gcn_rowptr + row + 1);
                for (int s_ = beg; s_ < end; ++s_) {
                    const float w0 = __ldg(p.ep.gcn_val + s_) * p.ep.gcn_scale;
                    const float* x0 = p.ep.gcn_x + (int64_t)__ldg(p.ep.gcn_idx + s_) * kDim + 32 * half;
                    float4 x[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) x[j] = ldg4(x0 + 4 * j);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        hs[4 * j] = fmaf(w0, x[j].x, hs[4 * j]); hs[4 * j + 1] = fmaf(w0, x[j].y, hs[4 * j + 1]);
                        hs[4 * j + 2] = fmaf(w0, x[j].z, hs[4 * j + 2]); hs[4 * j + 3] = fmaf(w0, x[j].w, hs[4 * j + 3]);
                    }
                }
            }
            if (p.ep.ln_weight != nullptr) {
                // LayerNorm over the 64 columns of the row = this thread's 32 + the partner's 32 (warp +-4, same lane): two-pass
                // statistics, each exchanged through shared memory under a 64-thread named barrier (id 1 + quad)
                float s1 = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) s1 += hs[j];
                ln_sum[half][lrow] = s1;
                bar_sync_named(1 + quad, 64);
                const float mean = (ln_sum[0][lrow] + ln_sum[1][lrow]) * (1.f / kDim);
                float s2 = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) { const float d_ = hs[j] - mean; s2 = fmaf(d_, d_, s2); }
                ln_var[half][lrow] = s2;
                bar_sync_named(1 + quad, 64);
                const float rstd = rsqrtf((ln_var[0][lrow] + ln_var[1][lrow]) * (1.f / kDim) + p.ep.ln_eps);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 w4 = ldg4(p.ep.ln_weight + 32 * half + j), b4 = ldg4(p.ep.ln_bias + 32 * half + j);
                    hs[j] = fmaf((hs[j] - mean) * rstd, w4.x, b4.x); hs[j + 1] = fmaf((hs[j + 1] - mean) * rstd, w4.y, b4.y);
                    hs[j + 2] = fmaf((hs[j + 2] - mean) * rstd, w4.z, b4.z); hs[j + 3] = fmaf((hs[j + 3] - mean) * rstd, w4.w, b4.w);
                }
            }
            if (p.ep.relu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) hs[j] = fmaxf(hs[j], 0.f);
            }
#pragma unroll
            for (int j = 0; j < 32; j += 4)
                sts128(obox + sw128(lane, j >> 2),
                       make_uint4(__float_as_uint(hs[j]), __float_as_uint(hs[j + 1]), __float_as_uint(hs[j + 2]), __float_as_uint(hs[j + 3])));
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                const int row0 = (int)(tile * kTile2) + quad * 32;
                if (p.store_hint) tma_store_2d_hint(&out_map, obox, 32 * half, row0, pol);
                else tma_store_2d(&out_map, obox, 32 * half, row0);
                tma_commit();
            }
            if (sc == H - 1 && ew == 0 && lane == 0) DIF_STAMP_ANY(p.dbg, 6);
        }
        if (ew == 0 && lane == 0) DIF_STAMP_ANY(p.dbg, 8);
        if (lane == 0) tma_wait_all0();      // stores must have landed before the CTA exits
    } else if (lane == 0) {
        // ===== MMA issuer (see apply_tc_kernel)
        const uint32_t idesc = make_idesc(kTile2, kBN, 0, 0);
        const uint32_t stage_base = smem_u32(stages), b_base = smem_u32(Bop);
        if (p.prepared != nullptr) mbar_wait(&bbar, 0);
        for (int st = 0; st < nst; ++st) {
            const int s = st % kNS2;
            const int sc0 = SHARED ? st * H : st;
            bool have_a = false;
#pragma unroll
            for (int hh = 0; hh < (SHARED ? H : 1); ++hh) {
                const int sc = sc0 + hh, slot = sc % kNAcc, h = sc % H;
                if (sc >= kNAcc) mbar_wait(&tempty[slot], ((sc / kNAcc) - 1) & 1);
                if (!have_a) { mbar_wait(&full[s], (st / kNS2) & 1); have_a = true; }
                tc_fence_after();
                const uint32_t sb = stage_base + s * kStage2, bb = b_base + h * 2 * kBOp;
                const uint32_t d = tmem + slot * kAccCols;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint64_t qhi = make_desc(sb + ks * 32, kKmajLBO, kKmajSBO), qlo = make_desc(sb + kQOp + ks * 32, kKmajLBO, kKmajSBO);
                    const uint64_t bhi = make_desc(bb + ks * 32, kKmajLBO, kKmajSBO), blo = make_desc(bb + kBOp + ks * 32, kKmajLBO, kKmajSBO);
                    umma(d, qhi, bhi, idesc, ks > 0 ? 1u : 0u);
                    umma(d, qlo, bhi, idesc, 1u);
                    umma(d, qhi, blo, idesc, 1u);
                }
                if (hh == (SHARED ? H : 1) - 1) umma_commit(&empty[s]);
                umma_commit(&tfull[slot]);
            }
        }
        DIF_STAMP_ANY(p.dbg, 7);
    }
    __syncwarp();
    if (warp == 0) DIF_STAMP(p.dbg, 3);
    tc_fence_before();
    __syncthreads();
    DIF_STAMP(p.dbg, 5);
    if (warp == 16) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------
// backward pass 2 (SURVEY.md 8a-1b): three streaming contractions with the same skeleton as apply_tc_kernel
//   KIND 0  dq = c (dnum S^T + dden z) - q t_q / sum q^2     A = g * (1/den)   B[n=m][k=d] = c S      rows from q
//   KIND 1  dk = c (v dS^T + dz)       - k t_k / sum k^2     A = v             B[n=m][k=d] = c dS     rows from k
//   KIND 2  dv = c  k dS + du                                A = k             B[n=d][k=m] = c dS^T
// ------------------------------------------------------------------------------------------
constexpr int kBOpB = 64 * 128;                       // one (head, hi|lo) B tile: 64 rows x 128 B
template <int H>
constexpr int smem_bwd_bytes() { return H * 2 * kBOpB + kNS2 * kStage2 + kOutStage + H * kDim * 4 + 1024; }

struct BwdTcArgs {
    const float* a_src;      // streamed into the A operand: g | v | k        [N,H,64]
    const float* e_src;      // epilogue row source: q | k | nullptr          [N,H,64]
    const float* rowscal;    // KIND 0: (1/den, dden) per (node, head)
    const float* fwd;        // forward partials  [S | z | u | sq | sk]
    const float* bwd;        // backward partials [dS | dz | du | t_q | t_k]
    int64_t N;
    float* out;
    int pf_tiles, store_hint;
};

template <int KIND, int H>
__global__ void __launch_bounds__(kThreadsTC, 1) bwd_apply_tc_kernel(const __grid_constant__ BwdTcArgs p, const __grid_constant__ CUtensorMap out_map,
                                                                         const __grid_constant__ CUtensorMap e_map) {
    using G = Geo<H>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* Bop = base;                                             // [h][hi|lo][64 rows][128 B]
    uint8_t* stages = base + H * 2 * kBOpB;
    uint8_t* ostage = stages + kNS2 * kStage2;
    float* vec = reinterpret_cast<float*>(ostage + kOutStage);       // [H][64]: c z | c dz | du
    __shared__ uint64_t full[kNS2], empty[kNS2], tfull[kNAcc], tempty[kNAcc], ebar[4];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t ntiles = (p.N + kTile2 - 1) / kTile2;
    const int my_tiles = blockIdx.x < ntiles ? (int)((ntiles - 1 - blockIdx.x) / gridDim.x + 1) : 0;
    const int nsc = my_tiles * H;
    auto tile_of = [&](int sc) -> int64_t { return blockIdx.x + (int64_t)(sc / H) * gridDim.x; };

    if (tid == 32 && my_tiles > 0) {
        for (int i = 0; i < 2 && i < my_tiles; ++i) {
            const int64_t prow = tile_of(H * i) * kTile2;
            const int64_t nrows = min((int64_t)kTile2, p.N - prow);
            for (int64_t r = 0; r < nrows; r += 16)
                prefetch_l2(p.a_src + (prow + r) * G::kRowF, (uint32_t)(min((int64_t)16, nrows - r) * G::kRowB));
        }
    }
    if (tid == 0) {
        for (int s = 0; s < kNS2; ++s) { mbar_init(&full[s], 8); mbar_init(&empty[s], 1); }
        for (int s = 0; s < kNAcc; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 4); }
        for (int s = 0; s < 4; ++s) mbar_init(&ebar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 12) tmem_alloc(&tmem_slot, 512);

    const float sq = p.fwd[G::offSq], sk = p.fwd[G::offSq + 1];
    const float c = 1.f / (sqrtf(sq) * sqrtf(sk));
    // coefficient of the epilogue row source: -t_q/sum q^2 (dq), -t_k/sum k^2 (dk)
    const float escale = KIND == 0 ? -p.bwd[G::offSq] / sq : (KIND == 1 ? -p.bwd[G::offSq + 1] / sk : 0.f);
    {
        // ---- B operands (K-major SW128, bf16 hi/lo, pre-scaled by c): row n, k-chunk ch
        const float* mat = KIND == 0 ? p.fwd : p.bwd;
        constexpr int kTasks = H * 8 * kDim, kPer = (kTasks + kThreadsTC - 1) / kThreadsTC;
        float x[kPer][8];
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int task = tid + u * kThreadsTC;
            const int n = task % kDim, hc = task / kDim, ch = hc & 7, h = hc >> 3;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int kk = ch * 8 + i;
                x[u][i] = 0.f;
                if (task < kTasks)
                    x[u][i] = KIND == 2 ? __ldg(mat + ((int64_t)h * kDim + kk) * kDim + n)      // B[n=d][k=m] = dS[m][d]
                                        : __ldg(mat + ((int64_t)h * kDim + n) * kDim + kk);     // B[n=m][k=d] = (d)S[m][d]
            }
        }
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int task = tid + u * kThreadsTC;
            if (task < kTasks) {
                const int n = task % kDim, hc = task / kDim, ch = hc & 7, h = hc >> 3;
#pragma unroll
                for (int i = 0; i < 8; ++i) x[u][i] *= c;
                uint4 hi, lo;
                split8(x[u], hi, lo);
                const uint32_t off = (uint32_t)(h * 2 * kBOpB) + sw128(n, ch);
                sts128(smem_u32(Bop) + off, hi);
                sts128(smem_u32(Bop) + kBOpB + off, lo);
            }
        }
        for (int i = tid; i < H * kDim; i += kThreadsTC)
            vec[i] = KIND == 0 ? p.fwd[G::offZ + i] * c : (KIND == 1 ? p.bwd[G::offZ + i] * c : p.bwd[G::offU + i]);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;

    if (warp < 8) {
        // ===== A producers (see apply_tc_kernel); KIND 0 scales the g rows by 1/den of their (node, head)
        float buf[2][4][8];
        auto issue = [&](int sc, int j, float (&dst)[8]) {
            if (sc >= nsc) return;
            const int64_t tile = tile_of(sc);
            const int t = tid + 256 * j, h = sc % H;
            const int64_t row = tile * kTile2 + (t >> 3);
            if (row < p.N) {
                ldg256_stream(p.a_src + row * G::kRowF + h * kDim + (t & 7) * 8, dst);
                if (KIND == 0) {
                    const float inv = __ldg(p.rowscal + (row * H + h) * 2);
#pragma unroll
                    for (int i = 0; i < 8; ++i) dst[i] *= inv;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[i] = 0.f;
            }
        };
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(0, j, buf[0][j]);
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(1, j, buf[1][j]);
        const uint32_t stage_base = smem_u32(stages);
        for (int sc = 0; sc < nsc; ++sc) {
            const int s = sc % kNS2;
            if (sc >= kNS2) mbar_wait(&empty[s], ((sc / kNS2) - 1) & 1);
            const uint32_t sb = stage_base + s * kStage2;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = tid + 256 * j;
                uint4 hi, lo;
                split8(buf[0][j], hi, lo);
                const uint32_t off = sw128(t >> 3, t & 7);
                sts128(sb + off, hi);
                sts128(sb + kQOp + off, lo);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int i = 0; i < 8; ++i) buf[0][j][i] = buf[1][j][i];
                issue(sc + 2, j, buf[1][j]);
            }
        }
    } else if (warp < 12) {
        // ===== epilogue: thread = one row; out = acc + vec (x dden for dq) + escale * row source.  The row source
        // (q or k rows of this tile/head) is TMA-loaded into the swizzled staging boxes, combined in place and the
        // boxes are TMA-stored: no scattered global access on the LSU in either direction.
        const int ew = warp - 8;
        const uint32_t obox = smem_u32(ostage) + ew * 2 * kOutBox;
        const uint64_t pol = policy_evict_first();
        for (int sc = 0; sc < nsc; ++sc) {
            const int64_t tile = tile_of(sc);
            const int h = sc % H, slot = sc % kNAcc;
            const int64_t row = tile * kTile2 + ew * 32 + lane;
            const bool ok = row < p.N;
            const int col = h * kDim, row0 = (int)(tile * kTile2) + ew * 32;
            if (lane == 0) {
                tma_wait_read0();                         // the previous store has finished reading the boxes
                if (KIND != 2) {
                    mbar_expect_tx(&ebar[ew], 2 * kOutBox);
                    tma_load_2d(obox, &e_map, col, row0, &ebar[ew]);
                    tma_load_2d(obox + kOutBox, &e_map, col + 32, row0, &ebar[ew]);
                }
            }
            __syncwarp();
            float vmul = 1.f;
            if (KIND == 0) vmul = ok ? __ldg(p.rowscal + (row * H + h) * 2 + 1) : 0.f;     // dden
            mbar_wait(&tfull[slot], (sc / kNAcc) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(ew * 32) << 16) + slot * kAccCols;
            if (KIND != 2) mbar_wait(&ebar[ew], sc & 1);
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
                for (int j = 0; j < 32; j += 4) {
                    const float4 v4 = *reinterpret_cast<const float4*>(vec + h * kDim + c0 + j);
                    const uint32_t saddr = obox + (c0 >> 5) * kOutBox + sw128(lane, j >> 2);
                    float4 e4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (KIND != 2) e4 = lds128(saddr);
                    float4 o;
                    o.x = fmaf(e4.x, escale, fmaf(v4.x, vmul, __uint_as_float(r[j])));
                    o.y = fmaf(e4.y, escale, fmaf(v4.y, vmul, __uint_as_float(r[j + 1])));
                    o.z = fmaf(e4.z, escale, fmaf(v4.z, vmul, __uint_as_float(r[j + 2])));
                    o.w = fmaf(e4.w, escale, fmaf(v4.w, vmul, __uint_as_float(r[j + 3])));
                    sts128(saddr, make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(o.w)));
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                if (p.store_hint) {
                    tma_store_2d_hint(&out_map, obox, col, row0, pol);
                    tma_store_2d_hint(&out_map, obox + kOutBox, col + 32, row0, pol);
                } else {
                    tma_store_2d(&out_map, obox, col, row0);
                    tma_store_2d(&out_map, obox + kOutBox, col + 32, row0);
                }
                tma_commit();
            }
        }
        if (lane == 0) tma_wait_all0();
    } else if (lane == 0) {
        // ===== MMA issuer: M=128, N=64, K=64: 4 K-steps x (hi*hi + lo*hi + hi*lo)
        const uint32_t idesc = make_idesc(kTile2, kDim, 0, 0);
        const uint32_t stage_base = smem_u32(stages), b_base = smem_u32(Bop);
        for (int sc = 0; sc < nsc; ++sc) {
            const int s = sc % kNS2, slot = sc % kNAcc, h = sc % H;
            if (p.pf_tiles > 0 && h == 0 && sc + H * p.pf_tiles < nsc) {
                const int64_t prow = tile_of(sc + H * p.pf_tiles) * kTile2;
                const int64_t nrows = min((int64_t)kTile2, p.N - prow);
                for (int64_t r = 0; r < nrows; r += 16)
                    prefetch_l2(p.a_src + (prow + r) * G::kRowF, (uint32_t)(min((int64_t)16, nrows - r) * G::kRowB));
            }
            if (sc >= kNAcc) mbar_wait(&tempty[slot], ((sc / kNAcc) - 1) & 1);
            mbar_wait(&full[s], (sc / kNS2) & 1);
            tc_fence_after();
            const uint32_t sb = stage_base + s * kStage2, bb = b_base + h * 2 * kBOpB;
            const uint32_t d = tmem + slot * kAccCols;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const uint64_t ahi = make_desc(sb + ks * 32, kKmajLBO, kKmajSBO), alo = make_desc(sb + kQOp + ks * 32, kKmajLBO, kKmajSBO);
                const uint64_t bhi = make_desc(bb + ks * 32, kKmajLBO, kKmajSBO), blo = make_desc(bb + kBOpB + ks * 32, kKmajLBO, kKmajSBO);
                umma(d, ahi, bhi, idesc, ks > 0 ? 1u : 0u);
                umma(d, alo, bhi, idesc, 1u);
                umma(d, ahi, blo, idesc, 1u);
            }
            umma_commit(&empty[s]);
            umma_commit(&tfull[slot]);
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 12) tmem_dealloc(tmem, 512);
}


// ------------------------------------------------------------------------------------------
// forward in ONE kernel: pass 1 -> grid-wide (and cross-GPU) sum -> pass 2, one cooperative persistent launch.
//
// Same pipelines as reduce_tma_kernel + apply_tc_kernel<0>, glued by the fused tail that already is a grid barrier:
//   * no second launch, prologue, TMEM allocation or kernel-boundary drain between the passes;
//   * pass 1 is split in two phases.  Phase A streams K and V only (TMA) and yields S, z, u and sum k^2: everything the
//     record / slice-sum / exchange / B-image tail needs.  Phase B streams Q (TMA, L2 evict_last) for sum q^2 alone, WHILE
//     the tail warps run that tail, so HBM stays busy through the grid-wide reduction.  sum q^2 only scales the epilogue
//     (c = 1/(|Q||K|)): it gets a grid round of its own (flags3, fused_sq_sum) that only the epilogue waits for.  With many
//     rows per CTA (FusedArgs::split_q = 0, see kSplitQRows) phase A streams Q together with K and V and phase B is empty;
//   * the Q producers of pass 2 start right after phase B; the MMA issuer fills the accumulator ring as soon as the B image
//     is in shared memory;
//   * a CTA applies pass 2 to the rows it streamed in phase B, last tile first: the Q rows it read most recently (L2
//     evict_last) are consumed while they are still resident.
// Warps: 0-7 converters -> Q phase B -> Q producers; 8-11 TMA issuer (warp 8) + tail -> epilogue; 12 MMA issuer of both passes.
// Shared memory: the two passes alias one dynamic allocation ([stg | ops] vs [Bop | Q stages | out staging | u]).  The
// phase-B ring lies behind Bop, so the B image may land over the phase-A staging ring while phase B still streams.
// ------------------------------------------------------------------------------------------
template <int H, bool W = false>
__global__ void __launch_bounds__(kThreadsTC, 1) simple_fused_kernel(const __grid_constant__ FusedArgs fa, const __grid_constant__ CUtensorMap out_map) {
    using G = Geo<H>;
    using P = PLay<H, W>;
    const ReduceArgs1& a = fa.r;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    // pass 1 view
    uint8_t* stg = base;
    uint8_t* ops = stg + G::kNSG * G::kStg;
    // pass 2 view
    uint8_t* Bop = base;                                             // [h][hi|lo][80 rows][128 B]
    uint8_t* stages = base + P::kBBytes;
    uint8_t* ostage = stages + kNS2 * kStage2;                       // [4 warps][2 boxes][32 rows][128 B], 1024-aligned
    float* us = reinterpret_cast<float*>(ostage + kOutStage);        // [H][64]
    __shared__ uint64_t sfull[G::kNSG], sempty[G::kNSG], ofull[G::kNO], oempty[G::kNO], done;
    __shared__ uint64_t full[kNS2], empty[kNS2], tfull[kNAcc], tempty[kNAcc], bbar;
    // phase B: a 64 KB Q staging ring behind the B image (over the pass-2 stages, idle until phase B ends): the B image may
    // land while phase B still streams.  64 KB in flight per SM keep HBM busy; 128 KB delay the tail's flag and slice loads
    // behind the queued bulk copies (barrier 1 ends 10 us later) and make the step slower.
    constexpr int kNQ = (64 << 10) / G::kStgT;
    static_assert(P::kBBytes + kNQ * G::kStgT <= smem_fused_bytes<H, W>() - 1024, "phase-B ring must fit behind the B image");
    uint8_t* qring = base + P::kBBytes;
    __shared__ uint64_t qfull[kNQ], qempty[kNQ];
    __shared__ uint32_t tmem_slot;
    __shared__ float part[16];
    __shared__ __align__(16) float red[H == 1 ? 64 * 65 : 2048];    // z / u partial sums of the converters, S halves (H == 1), fp64 chains of the tail
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t r0 = (int64_t)blockIdx.x * a.rows_per_cta;
    const int64_t r1 = min(a.N, r0 + (int64_t)a.rows_per_cta);
    const int iters = r1 > r0 ? (int)((r1 - r0 + G::kNodes - 1) / G::kNodes) : 0;
    const int my_tiles = r1 > r0 ? (int)((r1 - r0 + kTile2 - 1) / kTile2) : 0;
    const int nsc = my_tiles * H;                       // (tile, head) stages of pass 2
    auto row0_of = [&](int sc) -> int64_t { const int t = sc / H; return r0 + (int64_t)(fa.reverse ? my_tiles - 1 - t : t) * kTile2; };
    uint64_t* dbg = a.dbg;
    DIF_STAMP(dbg, 0);

    if (tid == 0) {
        for (int s = 0; s < G::kNSG; ++s) { mbar_init(&sfull[s], 1); mbar_init(&sempty[s], 8); }
        for (int s = 0; s < G::kNO; ++s) { mbar_init(&ofull[s], 8); mbar_init(&oempty[s], 1); }
        mbar_init(&done, 1);
        for (int s = 0; s < kNS2; ++s) { mbar_init(&full[s], 8); mbar_init(&empty[s], 1); }
        for (int s = 0; s < kNAcc; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 4); }
        mbar_init(&bbar, 1);
        for (int s = 0; s < kNQ; ++s) { mbar_init(&qfull[s], 1); mbar_init(&qempty[s], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 12) tmem_alloc(&tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    pdl_wait();                                         // programmatic dependent launch: everything above overlapped the previous kernel
    DIF_STAMP(dbg, 1);
    // flags3 epoch: same generation word as fused_tail (CTA 0 bumps it only after every CTA has published its record, i.e.
    // after every thread here has read it)
    const unsigned long long epoch3 =
        a.epoch + *reinterpret_cast<volatile unsigned long long*>(a.flags + (int64_t)gridDim.x * kFlagStride) * 0x9E3779B97F4A7C15ull + 2;
    float* rec = a.ws + (int64_t)blockIdx.x * a.ws_len;

    if (warp < 8) {
        // =================== pass 1, phase A: converters of K and V (+ Q unless fa.split_q) (see reduce_tma_kernel) ===================
        float zacc[4] = {0.f, 0.f, 0.f, 0.f}, uacc[4] = {0.f, 0.f, 0.f, 0.f};
        float ssk = 0.f, ssq = 0.f;
        {
            const uint32_t stg_base = smem_u32(stg), ops_base = smem_u32(ops);
            for (int it = 0; it < iters; ++it) {
                const int s = it % G::kNSG, o = it % G::kNO;
                const int nrows = (int)min((int64_t)G::kNodes, r1 - (r0 + (int64_t)it * G::kNodes));
                mbar_wait(&sfull[s], (it / G::kNSG) & 1);
                float4 x[G::kChunksPerThread][3];
#pragma unroll
                for (int i = 0; i < G::kChunksPerThread; ++i) {
                    const int u = tid + 256 * i, node = u / G::kChunksPerRow;
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
                        x[i][t] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (node < nrows && (t < 2 || !fa.split_q)) x[i][t] = lds128(stg_base + s * G::kStg + t * G::kStgT + u * 16);
                    }
                }
                if (it >= G::kNO) mbar_wait(&oempty[o], ((it / G::kNO) - 1) & 1);
                const uint32_t ob = ops_base + o * G::kOpStage;
#pragma unroll
                for (int i = 0; i < G::kChunksPerThread; ++i) {
                    const int u = tid + 256 * i, node = u / G::kChunksPerRow, cc = u % G::kChunksPerRow;
                    const int head = cc >> 4, m = (cc & 15) * 4;
                    const int blk = (H == 1) ? (node >> 4) : head;
                    const int kn = (H == 1) ? (node & 15) : node;
                    const uint32_t off = (uint32_t)(blk * G::kBlockTile + (kn >> 3) * 1024 + (kn & 7) * 128 +
                                                    ((((m >> 3) ^ kn) & 7) << 4) + ((m >> 2) & 1) * 8);
                    uint32_t hi[2], lo[2];
                    split4(x[i][0], hi, lo);
                    sts64(ob + 0 * G::kOp + off, hi[0], hi[1]);
                    sts64(ob + 1 * G::kOp + off, lo[0], lo[1]);
                    split4(x[i][1], hi, lo);
                    sts64(ob + 2 * G::kOp + off, hi[0], hi[1]);
                    sts64(ob + 3 * G::kOp + off, lo[0], lo[1]);
                    const float4 kk = x[i][0], vv = x[i][1], qq = x[i][2];
                    zacc[0] += kk.x; zacc[1] += kk.y; zacc[2] += kk.z; zacc[3] += kk.w;
                    uacc[0] += vv.x; uacc[1] += vv.y; uacc[2] += vv.z; uacc[3] += vv.w;
                    ssk = fmaf(kk.x, kk.x, ssk); ssk = fmaf(kk.y, kk.y, ssk); ssk = fmaf(kk.z, kk.z, ssk); ssk = fmaf(kk.w, kk.w, ssk);
                    ssq = fmaf(qq.x, qq.x, ssq); ssq = fmaf(qq.y, qq.y, ssq); ssq = fmaf(qq.z, qq.z, ssq); ssq = fmaf(qq.w, qq.w, ssq);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) { mbar_arrive(&ofull[o]); mbar_arrive(&sempty[s]); }
            }
        }
        // hand the column sums to the tail warps (static shared memory: nothing of pass 2 aliases it)
        ssk = warp_sum(ssk);
        if (lane == 0) part[warp] = ssk;
#pragma unroll
        for (int i = 0; i < 4; ++i) { red[tid * 4 + i] = zacc[i]; red[1024 + tid * 4 + i] = uacc[i]; }
        __threadfence_block();
        bar_arrive_named(1, 384);                      // barrier A: 256 arrivals here + the 128 tail threads' sync
        DIF_STAMP(dbg, 11);
        // =================== pass 1, phase B (fa.split_q): sum q^2 of the CTA's Q rows ===================
        // The stages are the pass-1 stages of the Q rows; thread tid visits their 16-byte chunks u = tid + 256 i, stage by stage,
        // exactly as the converters of reduce_tma_kernel do: the per-thread fma chains, the warp sums and the sum over warps are
        // bit-identical to its.  Thread 0 issues the bulk copies (L2 evict_last: pass 2 reads the rows again) into the kNQ-stage
        // ring once the last phase-A MMAs have released the operand ring the Q ring may overlap.
        if (fa.split_q) {
            const uint32_t qbase = smem_u32(qring);
            auto issue = [&](int it) {
                const int s = it % kNQ;
                const int64_t row = r0 + (int64_t)it * G::kNodes;
                const uint32_t bytes = (uint32_t)(min((int64_t)G::kNodes, r1 - row) * G::kRowB);
                mbar_expect_tx(&qfull[s], bytes);
                tma_load_1d_hint(qbase + s * G::kStgT, a.q + row * G::kRowF, bytes, &qfull[s], policy_evict_last());
            };
            if (tid == 0) {
                mbar_wait(&done, 0);
                for (int it = 0; it < kNQ && it < iters; ++it) issue(it);
            }
            __syncwarp();
            for (int it = 0; it < iters; ++it) {
                const int s = it % kNQ;
                const int nrows = (int)min((int64_t)G::kNodes, r1 - (r0 + (int64_t)it * G::kNodes));
                mbar_wait(&qfull[s], (it / kNQ) & 1);
#pragma unroll
                for (int i = 0; i < G::kChunksPerThread; ++i) {
                    const int u = tid + 256 * i, node = u / G::kChunksPerRow;
                    const float4 qq = node < nrows ? lds128(qbase + s * G::kStgT + u * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
                    ssq = fmaf(qq.x, qq.x, ssq); ssq = fmaf(qq.y, qq.y, ssq); ssq = fmaf(qq.z, qq.z, ssq); ssq = fmaf(qq.w, qq.w, ssq);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&qempty[s]);
                if (tid == 0 && it + kNQ < iters) {
                    mbar_wait(&qempty[s], (it / kNQ) & 1);
                    issue(it + kNQ);
                }
                __syncwarp();
            }
        }
        // publish sum q^2 (record + flags3).  The barrier also closes the phase-B ring: the pass-2 Q stages below alias it, so no
        // warp may store into them while another one still reads its last Q stage.
        ssq = warp_sum(ssq);
        if (lane == 0) part[8 + warp] = ssq;
        __threadfence_block();
        bar_sync_named(3, 256);
        if (tid == 0) {
            float sq = 0.f;
            for (int w = 0; w < 8; ++w) sq += part[8 + w];
            rec[P::offSq] = sq;
            asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(fa.flags3 + (int64_t)blockIdx.x * kFlagStride), "l"(epoch3) : "memory");
        }
        DIF_STAMP(dbg, 12);
        // without phase B, pass 1 may still read the operand ring of the LAST stages (MMAs pending): the Q stages of pass 2 alias
        // it, so the stores into shared memory wait for `done` (all MMAs complete); the register stages are loaded right away
        // =================== pass 2: Q producers (see apply_tc_kernel) ===================
        float buf[2][4][8];
        auto issue = [&](int sc, int j, float (&dst)[8]) {
            if (sc >= nsc) return;
            const int t = tid + 256 * j;
            const int64_t row = row0_of(sc) + (t >> 3);
            if (row < r1) {
                ldg256_stream(a.q + row * G::kRowF + (sc % H) * kDim + (t & 7) * 8, dst);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[i] = 0.f;
            }
        };
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(0, j, buf[0][j]);
#pragma unroll
        for (int j = 0; j < 4; ++j) issue(1, j, buf[1][j]);
        mbar_wait(&done, 0);
        DIF_STAMP(dbg, 3);
        const uint32_t stage_base = smem_u32(stages);
        for (int sc = 0; sc < nsc; ++sc) {
            const int s = sc % kNS2;
            if (sc >= kNS2) mbar_wait(&empty[s], ((sc / kNS2) - 1) & 1);
            const uint32_t sb = stage_base + s * kStage2;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = tid + 256 * j;
                uint4 hi, lo;
                split8(buf[0][j], hi, lo);
                const uint32_t off = sw128(t >> 3, t & 7);
                sts128(sb + off, hi);
                sts128(sb + kQOp + off, lo);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int i = 0; i < 8; ++i) buf[0][j][i] = buf[1][j][i];
                issue(sc + 2, j, buf[1][j]);
            }
        }
    } else if (warp < 12) {
        const int te = tid - 256, ew = warp - 8;        // 128 tail / epilogue threads
        if (warp == 8 && lane == 0) {
            // =================== pass 1, phase A: TMA issuer (K and V; Q too unless fa.split_q) ===================
            const uint32_t stg_base = smem_u32(stg);
            const uint64_t pol_first = policy_evict_first_(), pol_last = policy_evict_last();
            const int nt = fa.split_q ? 2 : 3;
            for (int it = 0; it < iters; ++it) {
                const int s = it % G::kNSG;
                if (it >= G::kNSG) mbar_wait(&sempty[s], ((it / G::kNSG) - 1) & 1);
                const int64_t row = r0 + (int64_t)it * G::kNodes;
                const uint32_t bytes = (uint32_t)(min((int64_t)G::kNodes, r1 - row) * G::kRowB);
                mbar_expect_tx(&sfull[s], nt * bytes);
                if (a.l2_hints) {
                    tma_load_1d_hint(stg_base + s * G::kStg + 0 * G::kStgT, a.k + row * G::kRowF, bytes, &sfull[s], pol_first);
                    tma_load_1d_hint(stg_base + s * G::kStg + 1 * G::kStgT, a.v + row * G::kRowF, bytes, &sfull[s], pol_first);
                    if (nt == 3) tma_load_1d_hint(stg_base + s * G::kStg + 2 * G::kStgT, a.q + row * G::kRowF, bytes, &sfull[s], pol_last);
                } else {
                    tma_load_1d(stg_base + s * G::kStg + 0 * G::kStgT, a.k + row * G::kRowF, bytes, &sfull[s]);
                    tma_load_1d(stg_base + s * G::kStg + 1 * G::kStgT, a.v + row * G::kRowF, bytes, &sfull[s]);
                    if (nt == 3) tma_load_1d(stg_base + s * G::kStg + 2 * G::kStgT, a.q + row * G::kRowF, bytes, &sfull[s]);
                }
            }
        }
        __syncwarp();
        // =================== tail (see reduce_tma_kernel): record, grid-wide slice sum (+ cross-GPU LL exchange) ===================
        mbar_wait(&done, 0);
        tc_fence_after();
        bar_sync_named(1, 384);                          // barrier A: the converters' column sums are in `red` / `part`
        if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 4] = gtime();
        for (int col = te; col < G::kRowF; col += 128) {
            float z = 0.f, u = 0.f;
            for (int t = col >> 2; t < 256; t += G::kChunksPerRow) { z += red[t * 4 + (col & 3)]; u += red[1024 + t * 4 + (col & 3)]; }
            rec[P::offZ + col] = z;
            rec[P::offU + col] = u;
        }
        if (te == 0) {
            float sk = 0.f;
            for (int w = 0; w < 8; ++w) sk += part[w];
            rec[P::offSq + 1] = sk;
        }
        if (H == 1) bar_sync_named(2, 128);              // `red` is re-used by the tail
        fused_tail<H, W, true>(a, fa.flags2, rec, te, ew, lane, tmem, iters > 0, red);
        if (te == 0) {
            mbar_expect_tx(&bbar, (uint32_t)P::kBBytes);
            for (int i = 0; i < P::kBTiles * 2; ++i)
                tma_load_1d(smem_u32(Bop) + i * kBOp, a.prepared + (size_t)i * kBOp, (uint32_t)kBOp, &bbar);
        }
        for (int i = te; i < H * kDim; i += 128) us[i] = __ldcg(a.partials + P::offU + i);
        const float sk = __ldcg(a.partials + P::offSq + 1);
        // the MMA issuer may fill the accumulator ring meanwhile: only the scaling below waits for sum q^2
        const float sq = fused_sq_sum<H, W>(a, fa.flags3, epoch3, te, red);     // ends with a 128-thread barrier: `us` is complete
        if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 13] = gtime();
        const float cscale = 1.f / (sqrtf(sq) * sqrtf(sk));
        // =================== pass 2: epilogue (see apply_tc_kernel) ===================
        const uint32_t obox = smem_u32(ostage) + ew * 2 * kOutBox;
        const uint64_t pol = policy_evict_first();
        float inv_den = 0.f;
        for (int sc = 0; sc < nsc; ++sc) {
            const int64_t trow = row0_of(sc);
            const int h = sc % H, slot = sc % kNAcc;
            mbar_wait(&tfull[slot], (sc / kNAcc) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(ew * 32) << 16) + slot * kAccCols;
            // wide: h = output half dh; the denominator column only exists in the dh = 0 accumulator and serves both halves
            if (!W || h == 0) {
                uint32_t qz_bits = tmem_ld1(taddr + kDim);
                tmem_ld_wait1(qz_bits);
                inv_den = 1.f / (fmaf(__uint_as_float(qz_bits), cscale, a.n_total));
            }
            if (lane == 0) tma_wait_read0();
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
                for (int j = 0; j < 32; j += 4) {
                    const float4 u4 = *reinterpret_cast<const float4*>(us + h * kDim + c0 + j);
                    float4 o;
                    o.x = fmaf(__uint_as_float(r[j]), cscale, u4.x) * inv_den;
                    o.y = fmaf(__uint_as_float(r[j + 1]), cscale, u4.y) * inv_den;
                    o.z = fmaf(__uint_as_float(r[j + 2]), cscale, u4.z) * inv_den;
                    o.w = fmaf(__uint_as_float(r[j + 3]), cscale, u4.w) * inv_den;
                    sts128(obox + (c0 >> 5) * kOutBox + sw128(lane, j >> 2),
                           make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(o.w)));
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                const int col = h * kDim;
                const int row0 = (int)trow + ew * 32;
                if (fa.store_hint) {
                    tma_store_2d_hint(&out_map, obox, col, row0, pol);
                    tma_store_2d_hint(&out_map, obox + kOutBox, col + 32, row0, pol);
                } else {
                    tma_store_2d(&out_map, obox, col, row0);
                    tma_store_2d(&out_map, obox + kOutBox, col + 32, row0);
                }
                tma_commit();
            }
        }
        if (lane == 0) tma_wait_all0();
    } else if (lane == 0) {
        // =================== MMA issuer: pass 1 ... ===================
        {
            const uint32_t idesc = make_idesc(128, 128, 1, 1);
            const uint32_t lbo = G::kBlockTile, sbo = 1024;
            const uint32_t ops_base = smem_u32(ops);
            for (int it = 0; it < iters; ++it) {
                const int o = it % G::kNO;
                mbar_wait(&ofull[o], (it / G::kNO) & 1);
                tc_fence_after();
                const uint32_t sb = ops_base + o * G::kOpStage;
#pragma unroll
                for (int p = 0; p < G::kPairs; ++p) {
                    const uint32_t ho = p * 2 * G::kBlockTile;
                    const uint64_t khi = make_desc(sb + 0 * G::kOp + ho, lbo, sbo), klo = make_desc(sb + 1 * G::kOp + ho, lbo, sbo);
                    const uint64_t vhi = make_desc(sb + 2 * G::kOp + ho, lbo, sbo), vlo = make_desc(sb + 3 * G::kOp + ho, lbo, sbo);
                    umma(tmem + p * 128, khi, vhi, idesc, it > 0 ? 1u : 0u);
                    umma(tmem + p * 128, khi, vlo, idesc, 1u);
                    umma(tmem + p * 128, klo, vhi, idesc, 1u);
                }
                umma_commit(&oempty[o]);
            }
            if (iters > 0) umma_commit(&done); else mbar_arrive(&done);
        }
        // =================== ... and pass 2 ===================
        const uint32_t idesc = make_idesc(kTile2, kBN, 0, 0);
        const uint32_t stage_base = smem_u32(stages), b_base = smem_u32(Bop);
        pdl_launch_dependents();                        // the next kernel of the stream may start its prologue as SMs free up
        mbar_wait(&bbar, 0);
        if (!W) {
            for (int sc = 0; sc < nsc; ++sc) {
                const int s = sc % kNS2, slot = sc % kNAcc, h = sc % H;
                if (sc >= kNAcc) mbar_wait(&tempty[slot], ((sc / kNAcc) - 1) & 1);
                mbar_wait(&full[s], (sc / kNS2) & 1);
                tc_fence_after();
                const uint32_t sb = stage_base + s * kStage2, bb = b_base + h * 2 * kBOp;
                const uint32_t d = tmem + slot * kAccCols;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint64_t qhi = make_desc(sb + ks * 32, kKmajLBO, kKmajSBO), qlo = make_desc(sb + kQOp + ks * 32, kKmajLBO, kKmajSBO);
                    const uint64_t bhi = make_desc(bb + ks * 32, kKmajLBO, kKmajSBO), blo = make_desc(bb + kBOp + ks * 32, kKmajLBO, kKmajSBO);
                    umma(d, qhi, bhi, idesc, ks > 0 ? 1u : 0u);
                    umma(d, qlo, bhi, idesc, 1u);
                    umma(d, qhi, blo, idesc, 1u);
                }
                umma_commit(&empty[s]);
                umma_commit(&tfull[slot]);
            }
        } else {
            // wide: stage sc = (tile, K block kb); accumulator slot = (tile, output half dh) = the epilogue's stage index.
            // Both K blocks of a tile feed both halves: 2 x 2 x 4 K steps x 3 MMAs per tile.
            for (int sc = 0; sc < nsc; sc += 2) {
                const int slot0 = sc % kNAcc, slot1 = (sc + 1) % kNAcc;
                if (sc >= kNAcc) {
                    mbar_wait(&tempty[slot0], ((sc / kNAcc) - 1) & 1);
                    mbar_wait(&tempty[slot1], (((sc + 1) / kNAcc) - 1) & 1);
                }
#pragma unroll
                for (int kb = 0; kb < 2; ++kb) {
                    const int st_ = sc + kb, s = st_ % kNS2;
                    mbar_wait(&full[s], (st_ / kNS2) & 1);
                    tc_fence_after();
                    const uint32_t sb = stage_base + s * kStage2;
#pragma unroll
                    for (int dh = 0; dh < 2; ++dh) {
                        const uint32_t bb = b_base + (2 * dh + kb) * 2 * kBOp;
                        const uint32_t d = tmem + (dh == 0 ? slot0 : slot1) * kAccCols;
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint64_t qhi = make_desc(sb + ks * 32, kKmajLBO, kKmajSBO), qlo = make_desc(sb + kQOp + ks * 32, kKmajLBO, kKmajSBO);
                            const uint64_t bhi = make_desc(bb + ks * 32, kKmajLBO, kKmajSBO), blo = make_desc(bb + kBOp + ks * 32, kKmajLBO, kKmajSBO);
                            umma(d, qhi, bhi, idesc, (kb > 0 || ks > 0) ? 1u : 0u);
                            umma(d, qlo, bhi, idesc, 1u);
                            umma(d, qhi, blo, idesc, 1u);
                        }
                    }
                    umma_commit(&empty[s]);
                }
                umma_commit(&tfull[slot0]);
                umma_commit(&tfull[slot1]);
            }
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    DIF_STAMP(dbg, 7);
    if (warp == 12) tmem_dealloc(tmem, 512);
}

}  // namespace (kernels)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// fp32 [rows][cols] row-major tensor, box = 32 rows x 32 floats (128 B), 128B swizzle.
// cuTensorMapEncodeTiled is a driver call (tens of microseconds): encoded maps are cached per (base, rows, cols) --
// the caching allocator hands the same addresses back every step, so steady-state calls do not encode at all.
int make_out_map_uncached(CUtensorMap* map, float* base, int64_t rows, int64_t cols);

int make_out_map(CUtensorMap* map, float* base, int64_t rows, int64_t cols) {
    struct Key { float* b; int64_t r, c; };
    struct Entry { Key k; CUtensorMap m; };
    static std::mutex mu;
    static std::vector<Entry> cache;
    {
        std::lock_guard<std::mutex> lk(mu);
        for (const Entry& e : cache)
            if (e.k.b == base && e.k.r == rows && e.k.c == cols) { *map = e.m; return DIF_OK; }
    }
    int rc = make_out_map_uncached(map, base, rows, cols);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(mu);
    if (cache.size() >= 64) cache.erase(cache.begin());
    cache.push_back(Entry{Key{base, rows, cols}, *map});
    return DIF_OK;
}

int make_out_map_uncached(CUtensorMap* map, float* base, int64_t rows, int64_t cols) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        DIF_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q));
        DIF_REQUIRE(f && q == cudaDriverEntryPointSuccess, DIF_ECUDA, "cuTensorMapEncodeTiled not available in this driver");
        fn = (EncodeTiledFn)f;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)cols * 4};
    const cuuint32_t box[2] = {32, 32}, estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    DIF_REQUIRE(r == CUDA_SUCCESS, DIF_ECUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return DIF_OK;
}

bool simple_tc_supported(int64_t N, int H, int Hv, int M, int D) {
    return N >= 1 && (H == 1 || H == 2 || H == 4) && Hv == H && M == kDim && D == kDim;
}


int64_t simple_tc_workspace_bytes(int64_t N, int H, int Hv, int M, int D) {
    (void)Hv; (void)M; (void)D;
    int grid;
    tc_rows_per_cta(N, H, &grid);
    // per-CTA records + one 64-bit ready flag per CTA + the generation word
    return (int64_t)grid * tc_ws_len(H) * (int64_t)sizeof(float) + (int64_t)grid * 8 + 64;
}

int64_t simple_tc_prepared_bytes(int H, int Hv, int M, int D) {
    return simple_tc_supported(1, H, Hv, M, D) ? (int64_t)H * 2 * kBOp : 0;
}

template <int H, bool BWD>
static int launch_reduce(const ReduceArgs1& a, int grid, cudaStream_t st) {
    static bool attr_set = false;       // per (H, BWD) instantiation
    if (!attr_set) {
        DIF_CUDA_OK(cudaFuncSetAttribute(reduce_tma_kernel<H, BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, Geo<H>::kSmem1));
        attr_set = true;
    }
    void* args[] = {(void*)&a};
    // cooperative launch: the fused cross-CTA sum spins on per-CTA flags, so all CTAs must be co-resident
    // (grid <= #SMs, 1 CTA/SM); the runtime refuses the launch otherwise instead of deadlocking
    DIF_CUDA_OK(cudaLaunchCooperativeKernel((const void*)reduce_tma_kernel<H, BWD>, dim3(grid), dim3(kThreadsT), args, (size_t)Geo<H>::kSmem1, st));
    return DIF_OK;
}

int simple_reduce_tc(const float* q, const float* k, const float* v, int64_t N, int H, int Hv, int M, int D,
                     float* partials, void* prepared, void* ws, int64_t ws_bytes, cudaStream_t st,
                     void* const* peer_bufs, int rank, int world, unsigned long long seq, float* vbar) {
    DIF_REQUIRE(simple_tc_supported(N, H, Hv, M, D), DIF_EUNSUPPORTED, "tcgen05 path: unsupported shape");
    DIF_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v) & 15) == 0, DIF_EARG, "tcgen05 path: q/k/v must be 16-byte aligned");
    DIF_REQUIRE(prepared == nullptr || ((uintptr_t)prepared & 15) == 0, DIF_EARG, "simple_reduce(tcgen05): prepared buffer must be 16-byte aligned");
    int grid;
    const int rpc = tc_rows_per_cta(N, H, &grid);
    const int64_t ws_len = tc_ws_len(H);
    DIF_REQUIRE(ws_bytes >= (int64_t)grid * ws_len * 4 + (int64_t)(grid + 1) * 8, DIF_EARG, "simple_reduce(tcgen05): workspace too small");
    DIF_REQUIRE((((ws_len + kSlices - 1) / kSlices + 3) & ~(int64_t)3) <= kThreadsT, DIF_EUNSUPPORTED, "simple_reduce(tcgen05): slice wider than the CTA");
    static std::atomic<unsigned long long> epoch_src{0x9E3779B97F4A7C15ull ^ (unsigned long long)(uintptr_t)&epoch_src};
    ReduceArgs1 a{};
    a.q = q; a.k = k; a.v = v; a.N = N; a.rows_per_cta = rpc;
    a.ws = (float*)ws; a.ws_len = ws_len; a.flags = (unsigned long long*)((float*)ws + (int64_t)grid * ws_len);
    a.epoch = epoch_src.fetch_add(0x632BE59BD9B4E019ull) | 1ull;
    a.partials = partials; a.prepared = (uint8_t*)prepared;
    a.vbar = vbar;
    a.gram = (H == 1 && q == k && k == v) ? 1 : 0;
    static const int hints = env_int("DIF_TC_P1_HINTS", 1);
    a.l2_hints = hints;
    a.sh.world = 1;
    if (peer_bufs != nullptr && world > 1) {
        DIF_REQUIRE(world <= kCommMaxRanks && rank >= 0 && rank < world && seq > 0, DIF_EARG, "simple_reduce(sharded): bad rank/world/seq");
        for (int r = 0; r < world; ++r) { DIF_REQUIRE(peer_bufs[r], DIF_EARG, "simple_reduce(sharded): null peer buffer"); a.sh.bufs[r] = peer_bufs[r]; }
        a.sh.rank = rank; a.sh.world = world; a.sh.seq = seq;
        a.sh.lenpad = comm_lenpad(SimpleLayout{H, Hv, M, D}.len());
        a.sh.timeout_ns = comm_timeout_ns();
    }
    a.dbg = dbg_buffer();
    int rc = H == 4 ? launch_reduce<4, false>(a, grid, st) : H == 2 ? launch_reduce<2, false>(a, grid, st) : launch_reduce<1, false>(a, grid, st);
    if (rc) return rc;
    dbg_report("reduce_tma", a.dbg, grid);
    return DIF_OK;
}

template <int H, bool SHARED = false>
static int launch_apply(const ApplyTcArgs& a, const CUtensorMap& map, int grid, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        DIF_CUDA_OK(cudaFuncSetAttribute(apply_tc_kernel<H, SHARED>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2_bytes<H>()));
        attr_set = true;
    }
    apply_tc_kernel<H, SHARED><<<grid, kThreadsTC, smem2_bytes<H>(), st>>>(a, map);
    DIF_LAUNCH_OK();
    return DIF_OK;
}

template <int H, bool SHARED>
static int launch_layer(const ApplyTcArgs& a, const CUtensorMap& map, int grid, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        DIF_CUDA_OK(cudaFuncSetAttribute(layer_tc_kernel<H, SHARED>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2_bytes<H>()));
        attr_set = true;
    }
    layer_tc_kernel<H, SHARED><<<grid, kLayerThreads, smem2_bytes<H>(), st>>>(a, map);
    DIF_LAUNCH_OK();
    return DIF_OK;
}

int simple_apply_tc(const float* q, const float* partials, const void* prepared, double n_total, int64_t N, int H, int Hv, int M, int D,
                    float* out, const dif_epilogue_t* ep, cudaStream_t st, int64_t q_ld, int q_hs, const float* nvec) {
    DIF_REQUIRE(simple_tc_supported(N, H, Hv, M, D), DIF_EUNSUPPORTED, "tcgen05 path: unsupported shape");
    DIF_REQUIRE(((uintptr_t)q & 31) == 0 && ((uintptr_t)out & 15) == 0, DIF_EARG, "tcgen05 path: q must be 32-byte, out 16-byte aligned");
    DIF_REQUIRE(N < (1ll << 31), DIF_EUNSUPPORTED, "tcgen05 path: N must fit a 32-bit TMA coordinate");
    ApplyTcArgs a{};
    a.q = q; a.partials = partials; a.n_total = (float)n_total; a.N = N; a.out = out;
    a.q_ld = q_ld > 0 ? q_ld : (int64_t)H * kDim;
    a.q_hs = q_ld > 0 ? q_hs : kDim;
    a.nvec = nvec;
    DIF_REQUIRE((a.q_ld % 8) == 0 && (a.q_hs % 8) == 0, DIF_EARG, "simple_apply(tcgen05): row / head strides must be multiples of 8 floats");
    a.prepared = (const uint8_t*)prepared;
    DIF_REQUIRE(prepared == nullptr || ((uintptr_t)prepared & 15) == 0, DIF_EARG, "simple_apply(tcgen05): prepared buffer must be 16-byte aligned");
    if (ep) a.ep = *ep; else { a.ep = dif_epilogue_t{}; }
    DIF_REQUIRE(a.ep.mode == 0 || a.ep.mode == 1, DIF_EARG, "simple_apply: epilogue mode %d", a.ep.mode);
    DIF_REQUIRE(a.ep.gcn_rowptr == nullptr || (a.ep.mode == 1 && a.ep.gcn_idx && a.ep.gcn_val && a.ep.gcn_x && ((uintptr_t)a.ep.gcn_x & 15) == 0), DIF_EARG,
                "simple_apply: the in-epilogue gcn term needs mode 1 and rowptr / idx / val / x (x 16-byte aligned)");
    DIF_REQUIRE(a.ep.ln_weight == nullptr || (a.ep.ln_bias != nullptr && (((uintptr_t)a.ep.ln_weight | (uintptr_t)a.ep.ln_bias) & 15) == 0), DIF_EARG,
                "simple_apply: LayerNorm weight and bias must both be given, 16-byte aligned");
    static const int pf = env_int("DIF_TC_P2_PREFETCH", 1), sth = env_int("DIF_TC_P2_STORE_HINT", 1);
    a.pf_tiles = pf;
    a.store_hint = sth;
    a.dbg = dbg_buffer();
    const int grid = tc_grid((N + kTile2 - 1) / kTile2);
    CUtensorMap map;
    int rc = make_out_map(&map, out, N, a.ep.mode == 0 ? (int64_t)H * kDim : (int64_t)kDim);
    if (rc) return rc;
    static const int share = env_int("DIF_TC_P2_SHARED_A", 1);
    const bool shared_a = a.q_hs == 0 && H > 1 && share;            // one A operand for the H heads of a tile (projected form)
    if (a.ep.mode == 1) {       // layer epilogue: two threads per output row (layer_tc_kernel)
        rc = shared_a ? (H == 4 ? launch_layer<4, true>(a, map, grid, st) : launch_layer<2, true>(a, map, grid, st))
                      : (H == 4 ? launch_layer<4, false>(a, map, grid, st) : H == 2 ? launch_layer<2, false>(a, map, grid, st) : launch_layer<1, false>(a, map, grid, st));
    } else if (shared_a) {
        rc = H == 4 ? launch_apply<4, true>(a, map, grid, st) : launch_apply<2, true>(a, map, grid, st);
    } else {
        rc = H == 4 ? launch_apply<4>(a, map, grid, st) : H == 2 ? launch_apply<2>(a, map, grid, st) : launch_apply<1>(a, map, grid, st);
    }
    if (rc) return rc;
    dbg_report("apply_tc", a.dbg, grid);
    return DIF_OK;
}


// ---- forward in one kernel ----------------------------------------------------------------------
// ONE head of M = D = 128 (hidden_channels 128): the "wide" variant of the one-kernel forward (fp32 I/O)
bool simple_wide_supported(int64_t N, int H, int Hv, int M, int D) { return N >= 1 && H == 1 && Hv == 1 && M == 128 && D == 128; }

int64_t simple_fused_workspace_bytes(int64_t N, int H, int Hv, int M, int D) {
    const bool wide = simple_wide_supported(N, H, Hv, M, D);
    if (!wide && !simple_tc_supported(N, H, Hv, M, D)) return 0;
    int grid;
    tc_rows_per_cta(N, H, &grid);
    const int64_t ws_len = wide ? PLay<2, true>::kWsLen : tc_ws_len(H);
    return fused_ws_prepared_off(grid, ws_len) + (wide ? (int64_t)PLay<2, true>::kBBytes : (int64_t)H * 2 * kBOp) + 128;
}

template <int H, bool W = false>
static int launch_fused(const FusedArgs& a, const CUtensorMap& map, int grid, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        DIF_CUDA_OK(cudaFuncSetAttribute(simple_fused_kernel<H, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_fused_bytes<H, W>()));
        attr_set = true;
    }
    void* args[] = {(void*)&a, (void*)&map};
    return launch_persistent((const void*)simple_fused_kernel<H, W>, grid, kThreadsTC, (size_t)smem_fused_bytes<H, W>(), st, args);
}

// Q is streamed after K and V (phase B, overlapping the grid-wide reduction) when a CTA has at most this many rows.  The
// reduction takes ~20 us whatever N is: at 896 rows per CTA (N = 132 534) the overlap saves 10 us of a 133 us step; at 11 136
// rows (N = 1 632 803) it is a small share, and streaming K | V | Q together measured 55 us faster than the two phases (B200).
constexpr int kSplitQRows = 4096;

int simple_forward_tc(const float* q, const float* k, const float* v, int64_t N, int H, int Hv, int M, int D, double n_total,
                      float* partials, float* out, void* ws, int64_t ws_bytes, cudaStream_t st,
                      void* const* peer_bufs, int rank, int world, unsigned long long seq) {
    const bool wide = simple_wide_supported(N, H, Hv, M, D);
    DIF_REQUIRE(wide || simple_tc_supported(N, H, Hv, M, D), DIF_EUNSUPPORTED, "tcgen05 path: unsupported shape");
    DIF_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v) & 31) == 0 && ((uintptr_t)out & 15) == 0, DIF_EARG, "simple_forward: q/k/v must be 32-byte, out 16-byte aligned");
    DIF_REQUIRE(((uintptr_t)ws & 127) == 0, DIF_EARG, "simple_forward: workspace must be 128-byte aligned");
    DIF_REQUIRE(N < (1ll << 31), DIF_EUNSUPPORTED, "tcgen05 path: N must fit a 32-bit TMA coordinate");
    int grid;
    const int rpc = tc_rows_per_cta(N, H, &grid);
    const int64_t ws_len = wide ? PLay<2, true>::kWsLen : tc_ws_len(H);
    const int64_t poff = fused_ws_prepared_off(grid, ws_len);
    DIF_REQUIRE(ws_bytes >= poff + (wide ? (int64_t)PLay<2, true>::kBBytes : (int64_t)H * 2 * kBOp), DIF_EARG, "simple_forward: workspace too small");
    DIF_REQUIRE((((ws_len + kSlices - 1) / kSlices + 3) & ~(int64_t)3) <= 128, DIF_EUNSUPPORTED, "simple_forward: slice wider than the tail warps");
    static std::atomic<unsigned long long> epoch_src{0xA24BAED4963EE407ull ^ (unsigned long long)(uintptr_t)&epoch_src};
    FusedArgs fa{};
    ReduceArgs1& a = fa.r;
    a.q = q; a.k = k; a.v = v; a.N = N; a.rows_per_cta = rpc;
    a.ws = (float*)ws; a.ws_len = ws_len; a.flags = (unsigned long long*)((char*)ws + fused_ws_flags_off(grid, ws_len));
    fa.flags2 = a.flags + (int64_t)(grid + 1) * kFlagStride;
    fa.flags3 = fa.flags2 + (int64_t)grid * kFlagStride;
    a.epoch = epoch_src.fetch_add(0x632BE59BD9B4E019ull) | 1ull;
    a.partials = partials; a.prepared = (uint8_t*)ws + poff;
    a.vbar = nullptr;
    static const int hints = env_int("DIF_TC_P1_HINTS", 1), sth = env_int("DIF_TC_P2_STORE_HINT", 1), rev = env_int("DIF_TC_FUSED_REVERSE", 1);
    a.l2_hints = hints;
    fa.split_q = rpc <= kSplitQRows;
    a.n_total = (float)n_total;
    a.sh.world = 1;
    if (peer_bufs != nullptr && world > 1) {
        DIF_REQUIRE(world <= kCommMaxRanks && rank >= 0 && rank < world && seq > 0, DIF_EARG, "simple_forward(sharded): bad rank/world/seq");
        for (int r = 0; r < world; ++r) { DIF_REQUIRE(peer_bufs[r], DIF_EARG, "simple_forward(sharded): null peer buffer"); a.sh.bufs[r] = peer_bufs[r]; }
        a.sh.rank = rank; a.sh.world = world; a.sh.seq = seq;
        a.sh.lenpad = comm_lenpad(SimpleLayout{H, Hv, M, D}.len());
        a.sh.timeout_ns = comm_timeout_ns();
    }
    a.dbg = dbg_buffer();
    fa.out = out; fa.store_hint = sth; fa.reverse = rev;
    CUtensorMap map;
    int rc = make_out_map(&map, out, N, (int64_t)H * D);
    if (rc) return rc;
    rc = wide ? launch_fused<2, true>(fa, map, grid, st)
       : H == 4 ? launch_fused<4>(fa, map, grid, st) : H == 2 ? launch_fused<2>(fa, map, grid, st) : launch_fused<1>(fa, map, grid, st);
    if (rc) return rc;
    dbg_report("simple_fused", a.dbg, grid);
    return DIF_OK;
}

// ---- backward on the tensor cores -------------------------------------------------------------
int64_t simple_tc_rowscal_floats(int64_t N, int H) { return N * H * 2; }

int simple_bwd_reduce_tc(const float* q, const float* g, const float* out, const float* partials, double n_total,
                         int64_t N, int H, float* bwd_partials, float* rowscal, void* ws, int64_t ws_bytes, cudaStream_t st) {
    DIF_REQUIRE(simple_tc_supported(N, H, H, kDim, kDim), DIF_EUNSUPPORTED, "tcgen05 path: unsupported shape");
    DIF_REQUIRE((((uintptr_t)q | (uintptr_t)g | (uintptr_t)out) & 15) == 0 && ((uintptr_t)rowscal & 7) == 0, DIF_EARG, "tcgen05 bwd: misaligned pointer");
    int grid;
    const int rpc = tc_rows_per_cta(N, H, &grid);
    const int64_t ws_len = tc_ws_len(H);
    DIF_REQUIRE(ws_bytes >= (int64_t)grid * ws_len * 4 + (int64_t)(grid + 1) * 8, DIF_EARG, "simple_bwd_reduce(tcgen05): workspace too small");
    static std::atomic<unsigned long long> epoch_src{0xD1B54A32D192ED03ull ^ (unsigned long long)(uintptr_t)&epoch_src};
    ReduceArgs1 a{};
    a.k = q; a.v = g; a.q = out;                // roles: A <- q, B <- g (-> dnum), third stream <- out
    a.N = N; a.rows_per_cta = rpc;
    a.ws = (float*)ws; a.ws_len = ws_len; a.flags = (unsigned long long*)((float*)ws + (int64_t)grid * ws_len);
    a.epoch = epoch_src.fetch_add(0x632BE59BD9B4E019ull) | 1ull;
    a.partials = bwd_partials; a.prepared = nullptr;
    a.l2_hints = 0;
    a.sh.world = 1;
    a.fwd_partials = partials; a.n_total = (float)n_total; a.rowscal = rowscal;
    a.dbg = nullptr;
    return H == 4 ? launch_reduce<4, true>(a, grid, st) : H == 2 ? launch_reduce<2, true>(a, grid, st) : launch_reduce<1, true>(a, grid, st);
}

template <int KIND, int H>
static int launch_bwd_apply(const BwdTcArgs& a, int grid, cudaStream_t st) {
    CUtensorMap map, emap;
    int rc = make_out_map(&map, a.out, a.N, (int64_t)H * kDim);
    if (rc) return rc;
    if ((rc = make_out_map(&emap, const_cast<float*>(a.e_src ? a.e_src : a.a_src), a.N, (int64_t)H * kDim))) return rc;
    static bool attr_set = false;
    if (!attr_set) {
        DIF_CUDA_OK(cudaFuncSetAttribute(bwd_apply_tc_kernel<KIND, H>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bwd_bytes<H>()));
        attr_set = true;
    }
    bwd_apply_tc_kernel<KIND, H><<<grid, kThreadsTC, smem_bwd_bytes<H>(), st>>>(a, map, emap);
    DIF_LAUNCH_OK();
    return DIF_OK;
}

template <int H>
static int bwd_apply_all(BwdTcArgs a, const float* q, const float* k, const float* v, const float* g, float* dq, float* dk, float* dv,
                         int grid, cudaStream_t st) {
    int rc;
    a.a_src = g; a.e_src = q; a.out = dq;
    if ((rc = launch_bwd_apply<0, H>(a, grid, st))) return rc;
    a.a_src = v; a.e_src = k; a.out = dk;
    if ((rc = launch_bwd_apply<1, H>(a, grid, st))) return rc;
    a.a_src = k; a.e_src = nullptr; a.out = dv;
    return launch_bwd_apply<2, H>(a, grid, st);
}

int simple_bwd_apply_tc(const float* q, const float* k, const float* v, const float* g, const float* partials, const float* bwd_partials,
                        const float* rowscal, int64_t N, int H, float* dq, float* dk, float* dv, cudaStream_t st) {
    DIF_REQUIRE(simple_tc_supported(N, H, H, kDim, kDim), DIF_EUNSUPPORTED, "tcgen05 path: unsupported shape");
    DIF_REQUIRE(N < (1ll << 31), DIF_EUNSUPPORTED, "tcgen05 path: N must fit a 32-bit TMA coordinate");
    DIF_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)g) & 31) == 0 && (((uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) & 15) == 0,
                DIF_EARG, "tcgen05 bwd: misaligned pointer");
    BwdTcArgs a{};
    a.rowscal = rowscal; a.fwd = partials; a.bwd = bwd_partials; a.N = N;
    static const int pf = env_int("DIF_TC_P2_PREFETCH", 1), sth = env_int("DIF_TC_P2_STORE_HINT", 1);
    a.pf_tiles = pf;
    a.store_hint = sth;
    const int grid = tc_grid((N + kTile2 - 1) / kTile2);
    return H == 4 ? bwd_apply_all<4>(a, q, k, v, g, dq, dk, dv, grid, st)
         : H == 2 ? bwd_apply_all<2>(a, q, k, v, g, dq, dk, dv, grid, st)
                  : bwd_apply_all<1>(a, q, k, v, g, dq, dk, dv, grid, st);
}

}  // namespace dif
