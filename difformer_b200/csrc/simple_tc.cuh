// Shared by the tcgen05 'simple' kernels (simple_sm100.cu: fp32 I/O; simple_lp_sm100.cu: bf16 / fp16 I/O): compile-time
// geometry, kernel argument structs, host-side partition / workspace helpers and the fused tail that turns the per-CTA
// pass-1 records into the grid-wide (and cross-GPU) sum plus the pass-2 operand image inside a cooperative kernel.
#pragma once
#include <stdlib.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace dif {
namespace {

// ------------------------------------------------------------------------------------------
// compile-time geometry for H heads of 64 columns
// ------------------------------------------------------------------------------------------
template <int H>
struct Geo {
    static_assert(H == 1 || H == 2 || H == 4, "tcgen05 path: H in {1, 2, 4}");
    static constexpr int kRowF = H * kDim;              // floats per node row
    static constexpr int kRowB = kRowF * 4;             // bytes per node row
    // pass 1: the UMMA is M = N = 128 = two 64-wide MN blocks.  A block is a head (H >= 2) or, for H = 1, one of the
    // two 16-node halves of a 32-node stage (both halves accumulate S; the two diagonal blocks are added at the end).
    static constexpr int kBlocks = H < 2 ? 2 : H;
    static constexpr int kPairs = kBlocks / 2;
    static constexpr int kNodes = 16 * kBlocks / H;     // nodes per stage (32 for H = 1, else 16)
    static constexpr int kBlockTile = 16 * 128;         // [16 nodes][64 bf16]
    static constexpr int kOp = kBlocks * kBlockTile;    // one operand (Khi | Klo | Vhi | Vlo) of a stage
    static constexpr int kOpStage = 4 * kOp;
    static constexpr int kStgT = kNodes * kRowB;        // fp32 staging bytes of one tensor of a stage (= kBlocks * 4 KB)
    static constexpr int kStg = 3 * kStgT;              // K | V | Q
    static constexpr int kNSG = 3, kNO = 2;             // staging / operand ring depths
    static constexpr int kSmem1 = kNSG * kStg + kNO * kOpStage + 1024;
    static constexpr int kChunksPerRow = kRowB / 16;    // 16-byte chunks per node row (16 H)
    static constexpr int kChunksPerThread = kStgT / 16 / 256;   // = kBlocks (256 converter threads)
    static constexpr int kTmemCols1 = kPairs * 128 < 32 ? 32 : kPairs * 128;
    // partials layout [S | z | u | sq | sk]
    static constexpr int offZ = H * kDim * kDim, offU = offZ + H * kDim, offSq = offU + H * kDim, kP = offSq + 2;
    // pass 2
    static constexpr int kBBytes = H * 2 * 80 * 128;    // prepared B operands: per head hi | lo, 80 rows x 128 B
};

constexpr int kBOp = 80 * 128;                        // one (head, hi|lo) B-operand tile of pass 2

// Partials / B-image geometry of the one-kernel forward.  W ("wide") = ONE head of M = D = 128 (hidden_channels 128,
// run.sh:43,70,75) executed with the H = 2 geometry: the node rows have the same 512-byte layout, pass 1 is the very same
// M = N = 128 UMMA whose accumulator now is the whole S[128][128] (all four 64 x 64 blocks instead of the two diagonal ones),
// pass 2 contracts over K = 128 (two 64-column stages of Q) into the two 64-column halves of the output.
template <int H, bool W>
struct PLay {
    static_assert(!W || H == 2, "wide mode runs on the H = 2 geometry");
    static constexpr int kS = W ? 128 * 128 : H * kDim * kDim;          // floats of S
    static constexpr int kV = H * kDim;                                  // floats of z (= of u): 128 in wide mode
    static constexpr int offZ = kS, offU = offZ + kV, offSq = offU + kV, kP = offSq + 2;
    static constexpr int kBTiles = W ? 4 : H;                            // (head) or (output half dh, K block kb) tiles, each hi | lo
    static constexpr int kBBytes = kBTiles * 2 * kBOp;
    static constexpr int64_t kWsLen = (kP + 7) & ~7;                     // 32-byte aligned records (256-bit stores)
};
using ShardArgs = CommPeers;  // multi-GPU: peer-mapped LL exchange buffers (common.cuh, csrc/comm.cu)
constexpr int kThreadsT = 10 * 32;                    // pass 1: warps 0-7 converters, 8 TMA issuer, 9 MMA issuer
constexpr int kSlices = 148;                          // column slices of the record for the fused cross-CTA sum

struct ReduceArgs1 {
    const float *q, *k, *v;
    int64_t N;
    int rows_per_cta;
    float* ws;                    // per-CTA records [grid][ws_len]
    int64_t ws_len;
    unsigned long long* flags;    // [grid] record-ready flags
    unsigned long long epoch;
    float* partials;
    uint8_t* prepared;            // optional pass-2 operand image
    int l2_hints;
    ShardArgs sh;
    uint64_t* dbg;
    // backward (BWD): q -> A role, g -> B role (scaled to dnum = g/den on the fly), out -> third stream
    const float* fwd_partials;    // forward partials (S, z, u, sq, sk)
    float n_total;
    float* rowscal;               // [N][H][2] = (1/den, dden) per (node, head), consumed by the dq kernel
    float* vbar;                  // fwd, optional: mean over heads of V, [N][64] (feeds the gcn SpMM of the fused layer)
    int gram;                     // fwd, H = 1, q == k == v (Gram matrix of the layer input, projected.py): one stream instead of three
};


constexpr int kTile2 = 128;                           // rows per tile = UMMA M
constexpr int kQOp = kTile2 * 128;                    // 16 KB: [128 rows][64 bf16] of one head
constexpr int kStage2 = 2 * kQOp;                     // Qhi | Qlo
constexpr int kNS2 = 3;
constexpr int kBN = 80;                               // UMMA N: 64 columns of S + z column + padding
constexpr int kNAcc = 4, kAccCols = 128;              // TMEM accumulator ring (4 x 128 columns)
constexpr int kOutBox = 32 * 128;                     // TMA store box: 32 rows x 32 floats, 128B swizzle
constexpr int kOutStage = 4 * 2 * kOutBox;            // per epilogue warp: two boxes (column halves of a head)
template <int H>
constexpr int smem2_bytes() { return Geo<H>::kBBytes + kNS2 * kStage2 + kOutStage + H * kDim * 4 + 1024; }


struct FusedArgs {
    ReduceArgs1 r;            // pass 1 (+ tail, exchange) arguments; r.prepared = global scratch for the B-operand image (required)
    float* out;
    int store_hint, reverse;
    unsigned long long* flags2;   // [grid] second grid barrier (B image complete)
    unsigned long long* flags3;   // [grid] sum q^2 of the CTA is in its record
    int split_q;                  // 1: pass 1 reads Q after K and V (phase B, while the tail runs); 0: together with them
};
template <int H, bool W = false>
constexpr int smem_fused_bytes() {
    constexpr int p2 = PLay<H, W>::kBBytes + kNS2 * kStage2 + kOutStage + H * kDim * 4 + 1024;
    return Geo<H>::kSmem1 > p2 ? Geo<H>::kSmem1 : p2;
}

__device__ __forceinline__ void bar_sync_named(int id, int nthreads) { asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void bar_arrive_named(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(nthreads) : "memory"); }


int tc_grid(int64_t units) {
    const int sms = sm_count();
    return (int)(units < sms ? (units < 1 ? 1 : units) : sms);
}

// Row partition shared by both passes: contiguous ranges of whole 128-row tiles, one per CTA.
int tc_rows_per_cta(int64_t N, int H, int* grid) {
    (void)H;      // whole 128-row tiles per CTA: a multiple of the pass-1 stage (16 or 32 nodes) for every H
    int g = tc_grid((N + kTile2 - 1) / kTile2);
    int64_t rpc = (N + g - 1) / g;
    rpc = (rpc + kTile2 - 1) / kTile2 * kTile2;
    g = (int)((N + rpc - 1) / rpc);
    *grid = g;
    return (int)rpc;
}

// DIF_TC_DEBUG_TIMES=1: per-CTA %globaltimer stamps, summarised on stderr after a device sync (debug only)
uint64_t* dbg_buffer() {
    static uint64_t* buf = nullptr;
    static int on = -1;
    if (on < 0) { const char* e = getenv("DIF_TC_DEBUG_TIMES"); on = (e && atoi(e)) ? 1 : 0; }
    if (!on) return nullptr;
    if (!buf) cudaMalloc(&buf, 256 * kDbgSlots * sizeof(uint64_t));
    cudaMemset(buf, 0, 256 * kDbgSlots * sizeof(uint64_t));
    return buf;
}
void dbg_report(const char* name, uint64_t* buf, int grid) {
    if (!buf) return;
    cudaDeviceSynchronize();
    static uint64_t h[256 * kDbgSlots];
    cudaMemcpy(h, buf, sizeof(h), cudaMemcpyDeviceToHost);
    if (const char* path = getenv("DIF_TC_DEBUG_CSV")) {         // per-CTA stamps (slot 15 = %smid + 1) for offline analysis
        if (FILE* f = fopen(path, "a")) {
            for (int b = 0; b < grid; ++b) {
                fprintf(f, "%s,%d", name, b);
                for (int s_ = 0; s_ < kDbgSlots; ++s_) fprintf(f, ",%llu", (unsigned long long)h[b * kDbgSlots + s_]);
                fprintf(f, "\n");
            }
            fclose(f);
        }
    }
    uint64_t t0 = ~0ull;
    for (int b = 0; b < grid; ++b) if (h[b * kDbgSlots] && h[b * kDbgSlots] < t0) t0 = h[b * kDbgSlots];
    fprintf(stderr, "[%s] slot: min/avg/max us since first CTA start\n", name);
    for (int s = 0; s < kDbgSlots - 1; ++s) {
        double mn = 1e30, mx = 0, sum = 0; int n = 0;
        for (int b = 0; b < grid; ++b) { if (!h[b * kDbgSlots + s]) continue; double t = (h[b * kDbgSlots + s] - t0) * 1e-3; mn = t < mn ? t : mn; mx = t > mx ? t : mx; sum += t; ++n; }
        if (n) fprintf(stderr, "  stamp %d: %7.2f %7.2f %7.2f  (n=%d)\n", s, mn, sum / n, mx, n);
    }
}

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}


// Launch of a persistent kernel whose CTAs synchronise with each other through global flags (grid <= #SMs, 1 CTA/SM).
//   DIF_TC_LAUNCH=0 (default) cooperative launch: the runtime guarantees co-residency or refuses the launch
//   DIF_TC_LAUNCH=1           plain launch (co-resident in practice when nothing else occupies the SMs; checked once
//                             against the occupancy calculator) -- saves the cooperative-launch overhead
//   DIF_TC_LAUNCH=2           plain launch + programmatic dependent launch: the kernel's prologue (barrier init, TMEM
//                             allocation) overlaps the tail of the previous kernel in the stream; the kernels execute
//                             griddepcontrol.wait before their first global access
//   DIF_TC_LAUNCH=3           cooperative + programmatic dependent launch
// The plain modes are opt-in: two such kernels on two streams can each hold part of the SMs and wait for the rest forever;
// the cooperative launch is what rules that out.
inline int launch_persistent(const void* kernel, int grid, int threads, size_t smem, cudaStream_t st, void** args) {
    static const int mode = env_int("DIF_TC_LAUNCH", 0);
    static const int persist_mb = env_int("DIF_TC_L2_PERSIST_MB", -1);      // experiment: L2 set-aside for evict_last lines
    static bool persist_set = false;
    if (persist_mb >= 0 && !persist_set) {
        int dev = 0, mx = 0;
        DIF_CUDA_OK(cudaGetDevice(&dev));
        DIF_CUDA_OK(cudaDeviceGetAttribute(&mx, cudaDevAttrMaxPersistingL2CacheSize, dev));
        size_t want = (size_t)persist_mb << 20;
        if (want > (size_t)mx) want = (size_t)mx;
        fprintf(stderr, "[difformer_b200] persisting L2 set-aside: %zu MB (device maximum %d MB)\n", want >> 20, mx >> 20);
        DIF_CUDA_OK(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want));
        persist_set = true;
    }
    if (mode == 0) {
        DIF_CUDA_OK(cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(threads), args, smem, st));
        return DIF_OK;
    }
    if (mode == 3) {          // cooperative AND programmatic dependent launch (experiment: is the combination accepted?)
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr[2];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 2;
        DIF_CUDA_OK(cudaLaunchKernelExC(&cfg, kernel, args));
        return DIF_OK;
    }
    int nb = 0;
    DIF_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem));
    DIF_REQUIRE(nb >= 1 && grid <= sm_count(), DIF_ECUDA, "persistent kernel cannot be co-resident (grid %d, %d CTA/SM)", grid, nb);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = mode == 2 ? 1 : 0;
    DIF_CUDA_OK(cudaLaunchKernelExC(&cfg, kernel, args));
    return DIF_OK;
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

int64_t tc_ws_len(int H) { return (SimpleLayout{H, H, kDim, kDim}.len() + 7) & ~(int64_t)7; }   // 32-byte aligned records (256-bit stores)

// Grid-barrier flags of the one-kernel forward: one 128-byte line per CTA.  All CTAs poll all flags: with the flags packed 16 to
// a line, ~19 000 polling threads hammer ten L2 lines and the flag STORES queue behind the polls (measured: a 5 us barrier).
constexpr int kFlagStride = 16;      // u64 per flag slot
// workspace: [records grid x ws_len f32][pad to 128][flags (grid + 1) lines][flags2 grid lines][flags3 grid lines][B-operand image]
int64_t fused_ws_flags_off(int grid, int64_t ws_len) { return ((int64_t)grid * ws_len * 4 + 127) & ~(int64_t)127; }
int64_t fused_ws_prepared_off(int grid, int64_t ws_len) { return fused_ws_flags_off(grid, ws_len) + (int64_t)(3 * grid + 1) * kFlagStride * 8; }


// ------------------------------------------------------------------------------------------
// Fused tail of a one-kernel forward, executed by the 128 threads of the four tail / epilogue warps (te = 0..127,
// ew = warp % 4 = TMEM lane quadrant).  On entry: all pass-1 MMAs have completed and z, u, sum q^2, sum k^2 of this CTA
// are already in its record `rec`.  SQ_LATE: sum q^2 is not (it arrives later, see fused_sq_sum): that element is left out of
// the partials and of the cross-GPU exchange.  The function
//   1. drains the S accumulators (TMEM) into the record and publishes it (flag = epoch, release),
//   2. waits for every CTA's record (all CTAs are resident: 1 CTA/SM, grid <= #SMs), reads "its" column slices of all
//      records from L2 and sums them in a fixed order (fp64) -- deterministic, no float atomics,
//   3. multi-GPU: exchanges each slice with the peers (LL push over NVLink, common.cuh) and adds the ranks in rank order,
//   4. writes the reduced partials and the pass-2 B-operand image (bf16 hi/lo, 128B-swizzled, un-scaled) to global memory,
//   5. runs a second grid barrier (flags2) after which partials and image are complete and visible to every CTA.
// `red` : shared scratch, >= 64*65 floats when H == 1 (block halves of S), >= 1024 floats otherwise (chains of the slice sum).
// Uses named barrier 2 (128 threads).  No shared memory of the pipelines is touched: the Q prefetch of pass 2 may run.
// ------------------------------------------------------------------------------------------
// lane `l` of the polling warp waits until flags l, l + 32, ... (< grid, one per 128-byte line) all hold `epoch`, then fences (acquire)
__device__ __forceinline__ void poll_flags(const unsigned long long* flags, int grid, int l, unsigned long long epoch) {
    constexpr int kMax = 8;                               // grid <= 256
    bool ok;
    do {
        unsigned long long f[kMax];
#pragma unroll
        for (int i = 0; i < kMax; ++i) {
            const int r = l + 32 * i;
            f[i] = epoch;
            if (r < grid) asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(f[i]) : "l"(flags + (int64_t)r * kFlagStride) : "memory");
        }
        ok = true;
#pragma unroll
        for (int i = 0; i < kMax; ++i) ok = ok && f[i] == epoch;
    } while (!ok);
    __threadfence();
}

template <int H, bool W = false, bool SQ_LATE = false>
__device__ __forceinline__ void fused_tail(const ReduceArgs1& a, unsigned long long* flags2, float* rec, int te, int ew, int lane,
                                           uint32_t tmem, bool have_rows, float* red) {
    using G = Geo<H>;
    using P = PLay<H, W>;
    uint64_t* dbg = a.dbg;
    if (te == 0)
        for (int64_t i = P::kP; i < a.ws_len; ++i) rec[i] = 0.f;
    if (W) {
        // wide: the accumulator IS S[128][128]: warp quadrant ew holds rows m = 32 ew + lane, all 128 columns
        const int m = ew * 32 + lane;
#pragma unroll 1
        for (int cb = 0; cb < 4; ++cb) {
            uint32_t r[32];
            if (have_rows) {
                tmem_ld32(tmem + ((uint32_t)(ew * 32) << 16) + cb * 32, r);
                tmem_ld_wait32(r);
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) r[j] = 0u;
            }
            float* dst = rec + (int64_t)m * 128 + cb * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 8)
                asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                             :: "l"(dst + j), "r"(r[j]), "r"(r[j + 1]), "r"(r[j + 2]), "r"(r[j + 3]),
                                "r"(r[j + 4]), "r"(r[j + 5]), "r"(r[j + 6]), "r"(r[j + 7]) : "memory");
        }
    }
#pragma unroll 1
    for (int p = 0; p < (W ? 0 : G::kPairs); ++p) {
        const int wq = ew, hp = wq >> 1, m = (wq * 32 + lane) & 63;
        uint32_t r[2][32];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            if (have_rows) {
                tmem_ld32(tmem + ((uint32_t)(wq * 32) << 16) + p * 128 + hp * 64 + c * 32, r[c]);
                tmem_ld_wait32(r[c]);
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) r[c][j] = 0u;
            }
        }
        if (H == 1) {
            if (hp == 1) {
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int j = 0; j < 32; ++j) red[m * 65 + c * 32 + j] = __uint_as_float(r[c][j]);
            }
            bar_sync_named(2, 128);
            if (hp == 0) {
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[c][j] = __float_as_uint(__uint_as_float(r[c][j]) + red[m * 65 + c * 32 + j]);
            }
        }
        if (H != 1 || hp == 0) {
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
    tc_fence_before();
    __threadfence();
    bar_sync_named(2, 128);
    if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 5] = gtime();
    const int grid = gridDim.x;
    const unsigned long long gen = *reinterpret_cast<volatile unsigned long long*>(a.flags + (int64_t)grid * kFlagStride);
    const unsigned long long epoch = a.epoch + gen * 0x9E3779B97F4A7C15ull;
    if (te == 0) asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(a.flags + (int64_t)blockIdx.x * kFlagStride), "l"(epoch) : "memory");
    const int chunk = (int)((((a.ws_len + kSlices - 1) / kSlices) + 3) & ~(int64_t)3);
    const ShardArgs& sh = a.sh;
    const bool sharded = sh.world > 1;
    const int xslot = (int)(sh.seq & 1);
    if (sharded && blockIdx.x == 0 && te == 0) comm_check_status(sh);
    bool waited = false;
    double* gsum = reinterpret_cast<double*>(red);       // [3 groups][128] partial chains of the slice sum (3 KB of `red`)
    for (int sl = blockIdx.x; sl < kSlices; sl += grid) {
        const int64_t j0 = (int64_t)sl * chunk;
        const int slice = (int)max((int64_t)0, min(a.ws_len, j0 + chunk) - j0);
        if (slice <= 0) break;
        if (!waited) {
            // ONE warp polls (relaxed loads, one acquire fence after the last flag): few pollers, one flag per L2 line; a lane's
            // (up to 5) flags are loaded back to back -- one L2 round trip per polling round, not one per flag
            if (te < 32) poll_flags(a.flags, grid, te, epoch);
            bar_sync_named(2, 128);                      // every record is published and (through the acquiring threads) visible
            if (blockIdx.x == 0 && te == 0) *reinterpret_cast<volatile unsigned long long*>(a.flags + (int64_t)grid * kFlagStride) = gen + 1;
            waited = true;
            if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 8] = gtime();
        }
        // Slice sum.  Four groups of 32 threads; group g walks the records r = 4i + g (the four fixed chains of the sum), lane l
        // owns the four consecutive elements 4l..4l+3 of the slice and reads them as ONE 16-byte load per record straight from
        // L2 (ld.cg), 19 loads in flight: 2 L2 round trips for the whole slice at 148 records.  Chains are fp64 and are combined in the
        // fixed order (c0 + c1) + (c2 + c3): deterministic, identical to the two-launch path.
        {
            const int g = te >> 5, l = te & 31;
            double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
            if (4 * l < slice) {
                const float* col = a.ws + j0 + 4 * l;
                const int64_t ld = a.ws_len;
                const int gmain = grid & ~3;             // records beyond the last full group of four all belong to chain 0
                int r = g;
                for (; r + 4 * 18 < gmain; r += 4 * 19) {
                    float4 x[19];
#pragma unroll
                    for (int i = 0; i < 19; ++i) x[i] = __ldcg(reinterpret_cast<const float4*>(col + (int64_t)(r + 4 * i) * ld));
#pragma unroll
                    for (int i = 0; i < 19; ++i) { c0 += (double)x[i].x; c1 += (double)x[i].y; c2 += (double)x[i].z; c3 += (double)x[i].w; }
                }
                for (; r < gmain; r += 4) {
                    const float4 x = __ldcg(reinterpret_cast<const float4*>(col + (int64_t)r * ld));
                    c0 += (double)x.x; c1 += (double)x.y; c2 += (double)x.z; c3 += (double)x.w;
                }
                if (g == 0)
                    for (r = gmain; r < grid; ++r) {
                        const float4 x = __ldcg(reinterpret_cast<const float4*>(col + (int64_t)r * ld));
                        c0 += (double)x.x; c1 += (double)x.y; c2 += (double)x.z; c3 += (double)x.w;
                    }
            }
            if (g > 0) {
                double* d = gsum + (g - 1) * 128 + 4 * l;
                d[0] = c0; d[1] = c1; d[2] = c2; d[3] = c3;
            }
            bar_sync_named(2, 128);
            // group 0 holds chain 0 of its four elements in registers; hand the combined values to the element-owning threads
            if (g == 0 && 4 * l < slice) {
                const double* d = gsum + 4 * l;
                float* o = reinterpret_cast<float*>(gsum + 3 * 128);        // [128] floats behind the chains
                o[4 * l + 0] = (float)((c0 + d[0]) + (d[128 + 0] + d[256 + 0]));
                o[4 * l + 1] = (float)((c1 + d[1]) + (d[128 + 1] + d[256 + 1]));
                o[4 * l + 2] = (float)((c2 + d[2]) + (d[128 + 2] + d[256 + 2]));
                o[4 * l + 3] = (float)((c3 + d[3]) + (d[128 + 3] + d[256 + 3]));
            }
            bar_sync_named(2, 128);
        }
        const int64_t j = j0 + te;
        const bool live = te < slice && j < P::kP && !(SQ_LATE && j == P::offSq);
        const float local = live ? reinterpret_cast<const float*>(gsum + 3 * 128)[te] : 0.f;
        float sum = local;
        if (sharded && live) {
            const uint32_t tag = (uint32_t)sh.seq;
            for (int p = 1; p < sh.world; ++p) {
                int r = sh.rank + p;
                if (r >= sh.world) r -= sh.world;
                comm_ll_send(comm_ll_ptr(sh.bufs[r], sh.lenpad, xslot, sh.rank) + j, local, tag);
            }
            sum = comm_ll_sum(sh, xslot, j, tag, local);
        }
        if (live) {
            a.partials[j] = sum;
            if (j < P::offU) {
                // B tile t, row n (output column), k (contraction index) of this element.  Narrow: t = head.  Wide: t = 2 dh + kb
                // (dh = output half, kb = K block); the z column (row 64) lives in the dh = 0 tiles.
                int h, n, m;
                if (!W) {
                    if (j < P::offZ) { h = (int)(j >> 12); m = (int)(j >> 6) & 63; n = (int)j & 63; }
                    else { h = (int)(j - P::offZ) >> 6; m = (int)(j - P::offZ) & 63; n = kDim; }
                } else {
                    if (j < P::offZ) { const int mm = (int)(j >> 7), d = (int)j & 127; h = 2 * (d >> 6) + (mm >> 6); m = mm & 63; n = d & 63; }
                    else { const int mm = (int)(j - P::offZ); h = mm >> 6; m = mm & 63; n = kDim; }
                }
                const __nv_bfloat16 hi = __float2bfloat16_rn(sum);
                const __nv_bfloat16 lo = __float2bfloat16_rn(sum - __bfloat162float(hi));
                uint8_t* img = a.prepared + (size_t)h * 2 * kBOp + sw128(n, m >> 3) + (m & 7) * 2;
                *reinterpret_cast<__nv_bfloat16*>(img) = hi;
                *reinterpret_cast<__nv_bfloat16*>(img + kBOp) = lo;
            }
        }
    }
    if (blockIdx.x == grid - 1) {
        // rows 65..79 of every (tile, hi|lo) image are zero padding (N = 80 of the pass-2 UMMA); wide: the dh = 1 tiles have no
        // z row either (row 64)
        for (int i = te; i < P::kBTiles * 2 * 16 * 8; i += 128) {
            const int c = i & 7, rr = (i >> 3) % 16 + 64, t = i / (8 * 16);
            if (rr == 64 && !(W && (t >> 1) >= 2)) continue;           // t = 2 * tile + (hi|lo): tiles 2, 3 are dh = 1
            *reinterpret_cast<uint4*>(a.prepared + (size_t)t * kBOp + sw128(rr, c)) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    // ---- second grid barrier: the B-operand image and the partials are complete
    if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 9] = gtime();
    __threadfence();
    bar_sync_named(2, 128);
    const unsigned long long epoch2 = epoch + 1;
    if (te == 0) asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(flags2 + (int64_t)blockIdx.x * kFlagStride), "l"(epoch2) : "memory");   // ordered by the fence above
    if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 10] = gtime();
    if (te < 32) poll_flags(flags2, grid, te, epoch2);
    asm volatile("fence.proxy.async;" ::: "memory");
    bar_sync_named(2, 128);
    if (dbg != nullptr && te == 0) dbg[blockIdx.x * kDbgSlots + 6] = gtime();
}

// Grid-wide (and cross-GPU) sum q^2 for a fused_tail<SQ_LATE>, executed by the same 128 threads after it.  Every CTA has put its
// sum q^2 into the offSq element of its record and set its flags3 line to `epoch3`.  Every CTA sums the records itself, in the
// order of the slice sum of fused_tail (fp64 chains over records r = g mod 4, the records beyond the last full group of four in
// chain 0, combined as (c0 + c1) + (c2 + c3)), so the value is bit-identical to the one the two-launch path reduces.  Multi-GPU:
// CTA 0 pushes the local value to the peers' offSq LL words; every CTA polls them (comm_ll_sum does not consume them) and adds
// the ranks in rank order.  CTA 0 writes the result to the partials.  Returns the sum to every calling thread.
// `red`: shared scratch of >= 257 floats (grid <= 256).  Uses named barrier 2 (128 threads).
template <int H, bool W = false>
__device__ __forceinline__ float fused_sq_sum(const ReduceArgs1& a, const unsigned long long* flags3, unsigned long long epoch3, int te,
                                              float* red) {
    using P = PLay<H, W>;
    const int grid = gridDim.x;
    if (te < 32) {
        poll_flags(flags3, grid, te, epoch3);
        for (int r = te; r < grid; r += 32) red[r] = __ldcg(a.ws + (int64_t)r * a.ws_len + P::offSq);
        __syncwarp();
        const int gmain = grid & ~3;
        double c = 0.0;
        if (te < 4)
            for (int r = te; r < gmain; r += 4) c += (double)red[r];
        if (te == 0)
            for (int r = gmain; r < grid; ++r) c += (double)red[r];
        const double c1 = __shfl_sync(0xffffffffu, c, 1), c2 = __shfl_sync(0xffffffffu, c, 2), c3 = __shfl_sync(0xffffffffu, c, 3);
        __syncwarp();
        if (te == 0) {
            const float local = (float)((c + c1) + (c2 + c3));
            float sum = local;
            const ShardArgs& sh = a.sh;
            if (sh.world > 1) {
                const int xslot = (int)(sh.seq & 1);
                const uint32_t tag = (uint32_t)sh.seq;
                if (blockIdx.x == 0)
                    for (int p = 1; p < sh.world; ++p) {
                        int r = sh.rank + p;
                        if (r >= sh.world) r -= sh.world;
                        comm_ll_send(comm_ll_ptr(sh.bufs[r], sh.lenpad, xslot, sh.rank) + P::offSq, local, tag);
                    }
                sum = comm_ll_sum(sh, xslot, P::offSq, tag, local);
            }
            if (blockIdx.x == 0) a.partials[P::offSq] = sum;
            red[256] = sum;
        }
    }
    bar_sync_named(2, 128);
    return red[256];
}

}  // namespace
}  // namespace dif
