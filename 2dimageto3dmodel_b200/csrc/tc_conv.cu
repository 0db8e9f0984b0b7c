// Implicit-GEMM 2-D convolution on the 5th-generation tensor cores (sm_100a): the dense convs of the
// conv-GAN generator / discriminators (models/gan.py:57-65,163-177,294-302,359,364; SURVEY.md §8 a13/a14).
//
//   Y[n, y, x, co] = sum_t sum_ci  X[n, sy*y + dy[t], sx*x + dx[t], ci] * Wt[t, co, ci]      (NHWC, fp32)
//
// "Tap-shifted TMA" formulation: no im2col buffer.  A CTA owns 128 output pixels (a BW x BH x BI box of
// the output) x BN output channels.  For every filter tap t and every 32-channel slice of Cin the TMA
// producer issues ONE 4-D tiled load of the input box shifted by (dy[t], dx[t]) — out-of-bounds rows and
// columns are zero-filled by the TMA unit, which IS the convolution's zero padding — and one 3-D load of
// the weight slice; both land in 128-byte-swizzled K-major tiles that `tcgen05.mma.kind::tf32` consumes
// directly (fp32 words, tf32 precision, fp32 accumulation in TMEM).  The same kernel computes
//   * fprop   (dy = r - pad_y, dx = s, Wt[t] = W[:, :, r, s]),
//   * dgrad   (dy = pad_y - r, dx = -s, Wt[t] = W[:, :, r, s]^T)  — the "full" correlation falls out of the
//     TMA zero fill, and strided (4x4 / stride 2) dgrad runs as 4 parity classes with a strided epilogue,
//   * strided fprop (element strides in the tensor map).
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2-5 =
// epilogue (TMEM -> registers -> bias / LeakyReLU -> global).  STAGES-deep mbarrier ring between producer
// and MMA; tcgen05.commit frees a stage and finally signals the epilogue.
#include "tc_common.cuh"
#include "tc_rowwin.cuh"

namespace {

constexpr int BM = 128;         // output pixels per CTA  (UMMA M)
constexpr int BK = 32;          // fp32 channels per K slice = 128 B = one swizzle row
constexpr int UMMA_K = 8;       // tf32
constexpr int MAX_TAPS = 25;
constexpr int NTHREADS = 224;   // warp 0: A-operand TMA, warp 1: MMA issue, warps 2-5: epilogue, warp 6: B-operand TMA

struct ConvParams {
    int N, Hout, Wout, Cout;          // logical output extent covered by tiles (before the epilogue transform)
    int BW, BH, BI;                   // output box per CTA, BW*BH*BI == 128
    int tiles_x, tiles_y;             // tiles along W and H (tiles along N = gridDim.x / (tiles_x*tiles_y))
    int xbase;                        // first output column of this launch (a strip launch covers the last few columns)
    int ntaps, kslices;               // filter taps, Cin / 32
    int sy, sx;                       // input coordinate = s * out + d[t]
    int dy[MAX_TAPS], dx[MAX_TAPS];
    int wtap[MAX_TAPS];               // weight tap (row of the tap-major weight array) read for loop tap t
    // epilogue: out pixel (n, oy*y + ooy, ox*x + oox) of a tensor [N, OH, OW, OC], channel offset 0
    int OH, OW, OC, osy, osx, ooy, oox;
    float leaky;                      // 1.0 = identity
    int dbg_lbo, dbg_sbo, dbg_lt;     // MN-major descriptor offsets (bytes), layout type
    double* stats;                    // nullable: [2][Cout] fp64 sum / sum of squares of the (pre-bias) output, accumulated
    int fold;                         // > 0: the A operand is folded on the fly from a raw [N,H,W,8] tensor (thin stems): K slice ks
    int fold_y0;                      //      = image rows y + fold_y0 + 4 ks .. + 3 of the 8 channels (tensor map dims c, row, x, n)
    const float* mask;                // nullable: tensor of the output's geometry; acc *= (mask >= 0 ? 1 : mslope) before statistics / bias
    float mslope;                     //           (LeakyReLU adjoint fused into the input-gradient epilogue)
    int stats_sum;                    // statistics: sums only (the bias gradient of the fused adjoint)
    int ncls;                         // >= 1 output classes in ONE launch (the stride-2 input gradient's parity classes): class c uses taps
    int cooy[4], coox[4];             //      [c * ntaps, (c + 1) * ntaps) of dy / dx / wtap and the output offset (cooy[c], coox[c])
};

template <int BN, int STAGES>
struct Smem {
    static constexpr int A_BYTES = BM * BK * 4;
    static constexpr int B_BYTES = BN * BK * 4;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BN, int STAGES, bool WMN, int MINB>
__global__ void __launch_bounds__(NTHREADS, MINB)
conv_tf32_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                 const ConvParams p, const float* __restrict__ bias, float* __restrict__ out) {
    using S = Smem<BN, STAGES>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(base + STAGES * S::STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* acc_full = empty + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // tile coordinates
    int t = blockIdx.x;
    const int tx = t % p.tiles_x;
    t /= p.tiles_x;
    const int ty = t % p.tiles_y;
    const int tn = t / p.tiles_y;
    const int x0 = p.xbase + tx * p.BW, y0 = ty * p.BH, n0 = tn * p.BI;
    const int c0 = blockIdx.y * BN;

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmap_x);
        tc::tma_prefetch_desc(&tmap_w);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(full + s, 1);
            tc::mbar_init(empty + s, 1);
        }
        tc::mbar_init(acc_full, 1);
        tc::fence_barrier_init();
    }
    if (warp == 2) tc::tmem_alloc<(BN < 32 ? 32 : BN)>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;
    const int KI = p.ntaps * p.kslices;

    // One elected lane spends ~200 cycles per TMA instruction (profiles/r1_conv_layers.md), about the tensor-core time of
    // the K slice it feeds, so the two operands are issued by two different warps; both complete on the same barrier.
    if (warp == 0) {
        if (lane == 0) {
            for (int it = 0; it < KI; ++it) {
                const int s = it % STAGES, ph = (it / STAGES) & 1;
                tc::mbar_wait(empty + s, ph ^ 1);
                const int tap = it / p.kslices, ks = it % p.kslices;
                unsigned char* a = base + s * S::STAGE_BYTES;
                tc::mbar_arrive_expect_tx(full + s, S::STAGE_BYTES);
                tc::tma_load_4d(a, &tmap_x, full + s, ks * BK, p.sx * x0 + p.dx[tap], p.sy * y0 + p.dy[tap], n0);
            }
        }
    } else if (warp == 6) {
        if (lane == 0) {
            for (int it = 0; it < KI; ++it) {
                const int s = it % STAGES, ph = (it / STAGES) & 1;
                tc::mbar_wait(empty + s, ph ^ 1);
                const int tap = it / p.kslices, ks = it % p.kslices;
                unsigned char* b = base + s * S::STAGE_BYTES + S::A_BYTES;
                if constexpr (WMN) {      // weights [tap][Cin][Cout]: 32 cin rows x 32 cout per box (N-major B operand)
#pragma unroll
                    for (int nb = 0; nb < BN / 32; ++nb) tc::tma_load_3d(b + nb * 4096, &tmap_w, full + s, c0 + nb * 32, ks * BK, p.wtap[tap]);
                } else {
                    tc::tma_load_3d(b, &tmap_w, full + s, ks * BK, c0, p.wtap[tap]);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = tc::umma_idesc_tf32(BM, BN, false, WMN);
            for (int it = 0; it < KI; ++it) {
                const int s = it % STAGES, ph = (it / STAGES) & 1;
                tc::mbar_wait(full + s, ph);
                tc::tc_fence_after();
                const uint32_t a = tc::smem_u32(base + s * S::STAGE_BYTES);
                const uint32_t b = a + S::A_BYTES;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t da = tc::umma_desc_k128(a + k * UMMA_K * 4);
                    const uint64_t db = WMN ? tc::umma_desc_mn128(b + k * 1024, p.dbg_lbo, p.dbg_sbo, p.dbg_lt) : tc::umma_desc_k128(b + k * UMMA_K * 4);
                    tc::umma_tf32(tmem_acc, da, db, idesc, (it | k) ? 1u : 0u);
                }
                tc::umma_commit(empty + s);          // frees the stage when these MMAs have read it
            }
            tc::umma_commit(acc_full);               // accumulator complete
        }
    } else {
        // epilogue warps 2..5: TMEM lane quarter = warp % 4
        const int q = warp & 3;
        const int r = q * 32 + lane;                 // row of the tile = output pixel
        const int bx = r % p.BW, by = (r / p.BW) % p.BH, bi = r / (p.BW * p.BH);
        const int n = n0 + bi, y = y0 + by, x = x0 + bx;
        const bool valid = n < p.N && y < p.Hout && x < p.Wout;
        float* dst = out + (((size_t)n * p.OH + (size_t)(p.osy * y + p.ooy)) * p.OW + (size_t)(p.osx * x + p.oox)) * p.OC;
        tc::mbar_wait(acc_full, 0);
        tc::tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            tc::tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)c, v);
            if (valid) {
                const int cb = c0 + c;
                if (cb + 32 <= p.Cout && (p.OC & 3) == 0) {       // full 32-channel run: 8 x 16-byte stores
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float4 o;
                        o.x = v[j] + (bias ? __ldg(bias + cb + j) : 0.f);
                        o.y = v[j + 1] + (bias ? __ldg(bias + cb + j + 1) : 0.f);
                        o.z = v[j + 2] + (bias ? __ldg(bias + cb + j + 2) : 0.f);
                        o.w = v[j + 3] + (bias ? __ldg(bias + cb + j + 3) : 0.f);
                        o.x = o.x >= 0.f ? o.x : o.x * p.leaky;
                        o.y = o.y >= 0.f ? o.y : o.y * p.leaky;
                        o.z = o.z >= 0.f ? o.z : o.z * p.leaky;
                        o.w = o.w >= 0.f ? o.w : o.w * p.leaky;
                        *reinterpret_cast<float4*>(dst + cb + j) = o;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int co = cb + j;
                        if (co < p.Cout) {
                            float o = v[j] + (bias ? __ldg(bias + co) : 0.f);
                            dst[co] = o >= 0.f ? o : o * p.leaky;
                        }
                    }
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc<(BN < 32 ? 32 : BN)>(tmem_acc);
}

// ----------------------------------------------------------------------------------------------
// Persistent variant: one CTA loops over (tile, channel block) work items with TWO accumulators in tensor memory, so the
// epilogue of item j (TMEM -> registers -> global, then the store drain) overlaps the TMA / MMA main loop of item j+1
// inside the same CTA, and barrier init / TMEM allocation / descriptor prefetch are paid once per CTA instead of once
// per 128 output pixels.  ncu on the one-tile-per-CTA kernel (profiles/r1_c_conv_final_full.md): layers with short K
// loops (folded stems: 10 K slices, stride-2 dgrad classes: 16) keep the tensor pipe 18-23 % busy with no memory
// system above 60 % — the CTA lifetime is fill + epilogue + drain.
// Barriers: full/empty ring shared by all items (global K-slice counter), acc_full[2] (MMA -> epilogue, tcgen05.commit),
// acc_empty[2] (epilogue -> MMA, one arrival per epilogue warp).
// ----------------------------------------------------------------------------------------------
constexpr int PTHREADS = 192;   // warp 0: TMA, warp 1: MMA issue, warps 2-5: epilogue

// R = pixel tiles stacked per work item: they share every weight tile that arrives (R accumulators of BN columns per
// TMEM buffer), which cuts the weight bytes per FLOP through the L2 -> SM fabric by R.
template <int BN, int STAGES, int R>
struct PSmem {
    static constexpr int A_TILE = BM * BK * 4;
    static constexpr int A_BYTES = R * A_TILE;
    static constexpr int B_BYTES = BN * BK * 4;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 320 /*barriers*/ + 2 * BN * 4 /*BN statistics*/;
    static constexpr int CTAS_PER_SM = (2 * TOTAL <= 227 * 1024 && 4 * R * BN <= 512) ? 2 : 1;
};

template <int BN, int STAGES, bool WMN, int R>
__global__ void __launch_bounds__(PTHREADS, PSmem<BN, STAGES, R>::CTAS_PER_SM)
conv_tf32_persistent_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                            const ConvParams p, const float* __restrict__ bias, float* __restrict__ out, int tiles,
                            int groups, int work_items) {
    using S = PSmem<BN, STAGES, R>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(base + STAGES * S::STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* acc_full = empty + STAGES;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    float* sm_stats = reinterpret_cast<float*>(base + STAGES * S::STAGE_BYTES + 320);
    constexpr uint32_t TCOLS = 2 * R * BN < 32 ? 32 : 2 * R * BN;
    static_assert(TCOLS <= 512 && (TCOLS & (TCOLS - 1)) == 0, "TMEM: 2 buffers x R accumulators x BN columns");
    for (int i = threadIdx.x; i < 2 * BN; i += blockDim.x) sm_stats[i] = 0.f;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmap_x);
        tc::tma_prefetch_desc(&tmap_w);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(full + s, 1);
            tc::mbar_init(empty + s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            tc::mbar_init(acc_full + b, 1);
            tc::mbar_init(acc_empty + b, 4);
        }
        tc::fence_barrier_init();
    }
    if (warp == 2) tc::tmem_alloc<TCOLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;
    const int KI = p.ntaps * p.kslices;

    if (warp == 0) {
        {
            const uint32_t leader = tc::elect_one();          // convergent producer loop: one elected lane arrives / issues the copies
            uint32_t git = 0;
            for (int w = blockIdx.x; w < work_items; w += gridDim.x) {
                // classes are the fastest index: the CTAs that work on the same pixel tiles at the same time share them in L2
                const int cls = w % p.ncls, wq = w / p.ncls, tb = cls * p.ntaps;
                const int g = wq % groups, c0 = (wq / groups) * BN;
                int x0[R], y0[R], n0[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    int t = g * R + r;
                    t = t < tiles ? t : tiles - 1;           // a group past the end re-loads the last tile (its result is dropped)
                    x0[r] = p.xbase + (t % p.tiles_x) * p.BW;
                    t /= p.tiles_x;
                    y0[r] = (t % p.tiles_y) * p.BH;
                    n0[r] = (t / p.tiles_y) * p.BI;
                }
                for (int it = 0; it < KI; ++it, ++git) {
                    const int s = git % STAGES, ph = (git / STAGES) & 1;
                    tc::mbar_wait(empty + s, ph ^ 1);
                    const int tap = it / p.kslices, ks = it % p.kslices;
                    unsigned char* a = base + s * S::STAGE_BYTES;
                    unsigned char* b = a + S::A_BYTES;
                    tc::mbar_arrive_expect_tx_if(leader, full + s, S::STAGE_BYTES);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (p.fold)     // box {8 ch, BW px, 4 rows}: lands as [row][pixel][8 floats] = four 32-byte-swizzled K-step tiles
                            tc::tma_load_4d_if(leader, a + r * S::A_TILE, &tmap_x, full + s, 0, x0[r] + p.dx[tb + tap], y0[r] + p.fold_y0 + 4 * ks, n0[r]);
                        else
                            tc::tma_load_4d_if(leader, a + r * S::A_TILE, &tmap_x, full + s, ks * BK, p.sx * x0[r] + p.dx[tb + tap], p.sy * y0[r] + p.dy[tb + tap], n0[r]);
                    }
                    if constexpr (WMN) {
#pragma unroll
                        for (int nb = 0; nb < BN / 32; ++nb) tc::tma_load_3d_if(leader, b + nb * 4096, &tmap_w, full + s, c0 + nb * 32, ks * BK, p.wtap[tb + tap]);
                    } else {
                        tc::tma_load_3d_if(leader, b, &tmap_w, full + s, ks * BK, c0, p.wtap[tb + tap]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // convergent issue loop (tc_common.cuh "MMA issue from a CONVERGENT warp"): all lanes walk it, one elected lane issues
        const uint32_t leader = tc::elect_one();
        const uint32_t tmem_u = tc::warp_uniform(tmem_acc);
        constexpr uint32_t idesc = tc::umma_idesc_tf32(BM, BN, false, WMN);
        uint32_t git = 0, j = 0;
        for (int w = blockIdx.x; w < work_items; w += gridDim.x, ++j) {
            const uint32_t buf = j & 1;
            tc::mbar_wait(acc_empty + buf, ((j >> 1) & 1) ^ 1);      // the epilogue has drained this buffer
            tc::tc_fence_after();
            const uint32_t acc = tmem_u + buf * (R * BN);
            for (int it = 0; it < KI; ++it, ++git) {
                const int s = git % STAGES, ph = (git / STAGES) & 1;
                tc::mbar_wait(full + s, ph);
                tc::tc_fence_after();
                const uint32_t a = tc::smem_u32(base + s * S::STAGE_BYTES);
                const uint32_t b = a + S::A_BYTES;
                // on-the-fly fold: K step k = image row k of the 4-row box, a [128 px][32 B] tile of its own (32-byte swizzle)
                const uint64_t da0 = p.fold ? tc::umma_desc_k32(a) : tc::umma_desc_k128(a);
                const uint64_t db0 = WMN ? tc::umma_desc_mn128(b, p.dbg_lbo, p.dbg_sbo, p.dbg_lt) : tc::umma_desc_k128(b);
                const uint32_t astep = p.fold ? (BM * 32) >> 4 : (UMMA_K * 4) >> 4, bstep = WMN ? 1024 >> 4 : (UMMA_K * 4) >> 4;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
#pragma unroll
                    for (int r = 0; r < R; ++r)
                        tc::umma_tf32_words_if(leader, acc + r * BN, tc::desc_lo(da0) + r * (S::A_TILE >> 4) + k * astep, tc::desc_hi(da0),
                                               tc::desc_lo(db0) + k * bstep, tc::desc_hi(db0), idesc, (it | k) ? 1u : 0u);
                }
                tc::umma_commit_if(leader, empty + s);
            }
            tc::umma_commit_if(leader, acc_full + buf);
        }
    } else {
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const int bx = row % p.BW, by = (row / p.BW) % p.BH, bi = row / (p.BW * p.BH);
        uint32_t j = 0;
        for (int w = blockIdx.x; w < work_items; w += gridDim.x, ++j) {
            const int cls = w % p.ncls, wq = w / p.ncls;
            const int g = wq % groups, c0 = (wq / groups) * BN;
            const int ooy = p.cooy[cls], oox = p.coox[cls];
            const uint32_t buf = j & 1;
            constexpr int NW = R * (BN / 32);
            uint32_t mbits[NW];
            if (p.mask) {                                     // signs of the item's activation mask, fetched under its main loop
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    int t = g * R + r;
                    const bool tile_ok = t < tiles;
                    const int tx = t % p.tiles_x;
                    t /= p.tiles_x;
                    const int n = (t / p.tiles_y) * p.BI + bi, y = (t % p.tiles_y) * p.BH + by, x = p.xbase + tx * p.BW + bx;
                    const bool valid = tile_ok && n < p.N && y < p.Hout && x < p.Wout;
                    const size_t off = (((size_t)n * p.OH + (size_t)(p.osy * y + ooy)) * p.OW + (size_t)(p.osx * x + oox)) * p.OC;
#pragma unroll
                    for (int cc = 0; cc < BN / 32; ++cc) {
                        const int cb = c0 + 32 * cc;
                        mbits[r * (BN / 32) + cc] = (valid && cb < p.Cout)
                            ? tc::act_mask_bits32(p.mask + off + cb, cb + 32 <= p.Cout && (p.OC & 3) == 0, p.Cout - cb) : 0xffffffffu;
                    }
                }
            }
            tc::mbar_wait(acc_full + buf, (j >> 1) & 1);
            tc::tc_fence_after();
#pragma unroll 1
            for (int r = 0; r < R; ++r) {
                int t = g * R + r;
                const bool tile_ok = t < tiles;
                const int tx = t % p.tiles_x;
                t /= p.tiles_x;
                const int n = (t / p.tiles_y) * p.BI + bi, y = (t % p.tiles_y) * p.BH + by, x = p.xbase + tx * p.BW + bx;
                const bool valid = tile_ok && n < p.N && y < p.Hout && x < p.Wout;
                const size_t off = (((size_t)n * p.OH + (size_t)(p.osy * y + ooy)) * p.OW + (size_t)(p.osx * x + oox)) * p.OC;
                float* dst = out + off;
#pragma unroll 1
                for (int c = 0; c < BN; c += 32) {
                    float v[32];
                    tc::tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + buf * (R * BN) + r * BN + (uint32_t)c, v);
                    if (r == R - 1 && c + 32 >= BN) {        // last read of this buffer: hand it back before the stores
                        tc::tc_fence_before();
                        __syncwarp();
                        if (lane == 0) tc::mbar_arrive(acc_empty + buf);
                    }
                    if (p.mask) tc::apply_act_bits32(v, tc::pick_word<NW>(mbits, r * (BN / 32) + c / 32), p.mslope);
                    if (p.stats) {
                        if (p.stats_sum) tc::stats_accumulate_sum(v, valid, sm_stats, c);
                        else tc::stats_accumulate(v, valid, sm_stats, BN, c);
                    }
                    if (valid) {
                        const int cb = c0 + c;
                        if (cb + 32 <= p.Cout && (p.OC & 3) == 0) {
#pragma unroll
                            for (int jj = 0; jj < 32; jj += 4) {
                                float4 o;
                                o.x = v[jj] + (bias ? __ldg(bias + cb + jj) : 0.f);
                                o.y = v[jj + 1] + (bias ? __ldg(bias + cb + jj + 1) : 0.f);
                                o.z = v[jj + 2] + (bias ? __ldg(bias + cb + jj + 2) : 0.f);
                                o.w = v[jj + 3] + (bias ? __ldg(bias + cb + jj + 3) : 0.f);
                                o.x = o.x >= 0.f ? o.x : o.x * p.leaky;
                                o.y = o.y >= 0.f ? o.y : o.y * p.leaky;
                                o.z = o.z >= 0.f ? o.z : o.z * p.leaky;
                                o.w = o.w >= 0.f ? o.w : o.w * p.leaky;
                                *reinterpret_cast<float4*>(dst + cb + jj) = o;
                            }
                        } else {
#pragma unroll
                            for (int jj = 0; jj < 32; ++jj) {
                                const int co = cb + jj;
                                if (co < p.Cout) {
                                    float o = v[jj] + (bias ? __ldg(bias + co) : 0.f);
                                    dst[co] = o >= 0.f ? o : o * p.leaky;
                                }
                            }
                        }
                    }
                }
            }
            if (p.stats) tc::stats_flush(sm_stats, BN, p.stats, p.Cout, c0, threadIdx.x - 64);
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc<TCOLS>(tmem_acc);
}

// ----------------------------------------------------------------------------------------------
// wgrad:  dW[co, ci, r, s] += sum_{n,y,x} dY[n, y, x, co] * X[n, st*y + r - pad_y, st*x + s, ci]      (NHWC operands)
// GEMM with M = Cout (128), N = Cin (BN), K = output pixels.  In NHWC the reduction index (pixel) is the SLOW index
// of both operands, i.e. they are M/N-major: a K slice is a BWk x BHk box of 32 output pixels, loaded as 32-channel
// wide TMA boxes ([32 pixels][32 channels], CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) — four for dY, BN/32 for X, the X
// boxes shifted by the tap on the OUTER dims (zero fill = padding, element strides for stride 2).  tcgen05.mma reads
// them through MN-major shared-memory descriptors (layout SWIZZLE_128B_BASE32B — the 32-bit transpose layout: 4-row
// atoms, SBO 512 B, LBO 4096 B; plain SWIZZLE_128B yields zeros for tf32, measured), so no NCHW copy is ever made.
// One CTA per (co tile, ci tile, tap, K split); partial sums are reduced into dW with red.global.add.f32.
// ----------------------------------------------------------------------------------------------
struct WgradParams {
    int N, Hout, Wout, Cout, Cin;
    int BWk, BHk;                  // pixel box of one K slice, BWk * BHk == 32
    int kx, ky;                    // K slices along x and y per image
    int kh, kw, pad_y, st;
    int xoff;                      // the convolution reads x from column xoff on (a caller-side crop of the padded input)
    int splits;                    // K splits (gridDim.z / taps)
    int fold;                      // > 0: X is the raw stem input [N,H,W,8]; 32-"channel" block b = image rows y - fold_pad + 4b .. + 3
    int tapmajor;                  // dW layout: 0 = [Cout][Cin][kh][kw], 1 = tap-major [kh*kw][Cout][Cin] (the F layout)
    int tstep;                     // taps of one CTA are s0, s0 + tstep, ... (1: adjacent taps of a stride-1 conv,
                                   // 2: taps of equal parity of a stride-2 conv = adjacent rows of the strided window)
};

template <int BN, int T>
struct WgradSmem {
    static constexpr int A_BYTES = BM * BK * 4;
    static constexpr int B_BYTES = (BN / 32) * (T == 1 ? 32 : 36) * 128;
    static constexpr int STAGE_BYTES = ((A_BYTES + B_BYTES + 1023) / 1024) * 1024;
};

// T > 1: the CTA computes T horizontally adjacent taps (r, s0 .. s0+T-1) at once.  They share the dY tile, and their X
// operands are views of ONE staged window of 32 + T - 1 (rounded to 36) pixels shifted by s rows — T accumulators of BN
// columns in TMEM, ~T x fewer bytes per MAC through the L2 -> SM path that bounds this kernel (profiles/r1_conv_layers.md).
template <int BN, int STAGES, int T>
__global__ void __launch_bounds__(NTHREADS, (T * BN <= 256 && STAGES <= 4) ? 2 : 1)
wgrad_tf32_kernel(const __grid_constant__ CUtensorMap tmap_dy, const __grid_constant__ CUtensorMap tmap_x,
                  const WgradParams p, float* __restrict__ dw) {
    constexpr int BLK = BK * 32 * 4;                      // dY: one [32 pixels][32 channels] box = 4 KB
    constexpr int WROWS = T == 1 ? 32 : 36;               // X window rows (pixels) per 32-channel block
    constexpr int XBLK = WROWS * 128;
    using S = WgradSmem<BN, T>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(base + STAGES * S::STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* acc_full = empty + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int co0 = blockIdx.x * BM, ci0 = blockIdx.y * BN;
    const int gpr = p.kw / T;                             // tap groups per kernel row
    const int groups = p.kh * gpr;
    const int grp = blockIdx.z % groups, split = blockIdx.z / groups;
    const int r = grp / gpr, s = grp % gpr;               // first tap of the group (tstep 1: gpr is 1 or kw; tstep 2: parity)
    const int per_img = p.kx * p.ky;
    const long long ktotal = (long long)p.N * per_img;
    const long long k_lo = ktotal * split / p.splits, k_hi = ktotal * (split + 1) / p.splits;
    const int KI = (int)(k_hi - k_lo);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmap_dy);
        tc::tma_prefetch_desc(&tmap_x);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; ++i) {
            tc::mbar_init(full + i, 1);
            tc::mbar_init(empty + i, 1);
        }
        tc::mbar_init(acc_full, 1);
        tc::fence_barrier_init();
    }
    constexpr uint32_t TCOLS = T * BN <= 64 ? 64 : T * BN <= 128 ? 128 : T * BN <= 256 ? 256 : 512;
    if (warp == 2) tc::tmem_alloc<TCOLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;

    if (warp == 0 || warp == 6) {           // warp 0 streams dY, warp 6 streams X (two TMA issue lanes, one barrier)
        {
            const uint32_t leader = tc::elect_one();          // convergent producer loops: one elected lane arrives / issues the copies
            for (int it = 0; it < KI; ++it) {
                const int st = it % STAGES, ph = (it / STAGES) & 1;
                tc::mbar_wait(empty + st, ph ^ 1);
                const long long k = k_lo + it;
                const int n = (int)(k / per_img), rem = (int)(k % per_img);
                const int x0 = (rem % p.kx) * p.BWk, y0 = (rem / p.kx) * p.BHk;
                unsigned char* a = base + st * S::STAGE_BYTES;
                // channels are split as (32, C/32) in the tensor maps: ONE 5-D box lands all 32-channel blocks back to back
                if (warp == 0) {
                    tc::mbar_arrive_expect_tx_if(leader, full + st, S::STAGE_BYTES);
                    tc::tma_load_5d_if(leader, a, &tmap_dy, full + st, 0, x0, y0, n, co0 / 32);
                } else if (p.fold) {      // (c, row, x, n) boxes of 4 rows x 8 channels per pixel: one per 32-"channel" block
#pragma unroll
                    for (int blk = 0; blk < BN / 32; ++blk)
                        tc::tma_load_4d_if(leader, a + S::A_BYTES + blk * XBLK, &tmap_x, full + st, 0, y0 - p.pad_y + 4 * (ci0 / 32 + blk), x0 + s + p.xoff, n);
                } else {
                    tc::tma_load_5d_if(leader, a + S::A_BYTES, &tmap_x, full + st, 0, p.st * x0 + s + p.xoff, p.st * y0 + r - p.pad_y, n, ci0 / 32);
                }
            }
        }
    } else if (warp == 1) {
        // convergent issue loop (tc_common.cuh "MMA issue from a CONVERGENT warp"): all lanes walk it, one elected lane issues
        const uint32_t leader = tc::elect_one();
        const uint32_t tmem_u = tc::warp_uniform(tmem_acc);
        constexpr uint32_t idesc = tc::umma_idesc_tf32(BM, BN, true, true);
        for (int it = 0; it < KI; ++it) {
            const int st = it % STAGES, ph = (it / STAGES) & 1;
            tc::mbar_wait(full + st, ph);
            tc::tc_fence_after();
            const uint32_t a = tc::smem_u32(base + st * S::STAGE_BYTES);
            const uint64_t da0 = tc::umma_desc_mn128(a, BLK, 512), db0 = tc::umma_desc_mn128(a + S::A_BYTES, XBLK, 512);
#pragma unroll
            for (int t = 0; t < T; ++t)
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k)      // 8 pixel rows (two 4-row swizzle atoms, 1024 B) per MMA
                    tc::umma_tf32_words_if(leader, tmem_u + t * BN, tc::desc_lo(da0) + k * (1024 >> 4), tc::desc_hi(da0),
                                           tc::desc_lo(db0) + (((t + 8 * k) * 128) >> 4), tc::desc_hi(db0), idesc, (it | k) ? 1u : 0u);
            tc::umma_commit_if(leader, empty + st);
        }
        tc::umma_commit_if(leader, acc_full);
    } else if (KI > 0) {
        const int q = warp & 3;
        const int co = co0 + q * 32 + lane;
        tc::mbar_wait(acc_full, 0);
        tc::tc_fence_after();
#pragma unroll 1
        for (int t = 0; t < T; ++t)
#pragma unroll 1
            for (int c = 0; c < BN; c += 32) {
                float v[32];
                tc::tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(t * BN + c), v);
                if (co < p.Cout) {
                    if (p.tapmajor) {       // 32 consecutive input channels of one (tap, co) row: 8 x 16-byte reductions
                        float* row = dw + ((size_t)(r * p.kw + s + t * p.tstep) * p.Cout + co) * p.Cin + ci0 + c;
#pragma unroll
                        for (int j = 0; j < 32; j += 4)
                            if (ci0 + c + j < p.Cin) atomicAdd(reinterpret_cast<float4*>(row + j), make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int ci = ci0 + c + j;
                            if (ci < p.Cin) atomicAdd(dw + (((size_t)co * p.Cin + ci) * p.kh + r) * p.kw + s + t * p.tstep, v[j]);
                        }
                    }
                }
            }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc<TCOLS>(tmem_acc);
}

template <int BN, int STAGES, int T>
int launch_wgrad(const CUtensorMap& mdy, const CUtensorMap& mx, const WgradParams& p, float* dw, dim3 grid, cudaStream_t st) {
    constexpr int WROWS = T == 1 ? 32 : 36;
    constexpr int STAGE = ((BM * BK * 4 + (BN / 32) * WROWS * 128 + 1023) / 1024) * 1024;
    constexpr int TOTAL = STAGES * STAGE + 1024 + 256;
    static_assert(TOTAL <= 227 * 1024, "wgrad pipeline does not fit shared memory");
    B3D_CUDA_OK(cudaFuncSetAttribute(wgrad_tf32_kernel<BN, STAGES, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, TOTAL));
    wgrad_tf32_kernel<BN, STAGES, T><<<grid, NTHREADS, TOTAL, st>>>(mdy, mx, p, dw);
    B3D_LAUNCH_OK();
    b3d::add_variant("wgrad_tf32<%d,%d,%d>", BN, STAGES, T);
    return B3D_OK;
}

template <int BN, int STAGES, bool WMN, int MINB>
int launch(const CUtensorMap& mx, const CUtensorMap& mw, const ConvParams& p, const float* bias, float* out,
           int tiles, cudaStream_t st) {
    using S = Smem<BN, STAGES>;
    B3D_CUDA_OK(cudaFuncSetAttribute(conv_tf32_kernel<BN, STAGES, WMN, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     S::TOTAL));
    dim3 grid(tiles, b3d::ceil_div(p.Cout, BN));
    conv_tf32_kernel<BN, STAGES, WMN, MINB><<<grid, NTHREADS, S::TOTAL, st>>>(mx, mw, p, bias, out);
    B3D_LAUNCH_OK();
    b3d::add_variant("conv_tf32<%d,%d,%d,%d>", BN, STAGES, (int)WMN, MINB);
    return B3D_OK;
}

template <int BN, int STAGES, bool WMN, int R>
int launch_persistent(const CUtensorMap& mx, const CUtensorMap& mw, const ConvParams& p, const float* bias, float* out,
                      int tiles, cudaStream_t st) {
    using S = PSmem<BN, STAGES, R>;
    static_assert(S::TOTAL <= 227 * 1024, "persistent conv pipeline does not fit shared memory");
    B3D_CUDA_OK(cudaFuncSetAttribute(conv_tf32_persistent_kernel<BN, STAGES, WMN, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    const int groups = b3d::ceil_div(tiles, R);
    const int work = groups * b3d::ceil_div(p.Cout, BN) * p.ncls;
    const int slots = S::CTAS_PER_SM * 148;
    const int grid = work < slots ? work : slots;
    conv_tf32_persistent_kernel<BN, STAGES, WMN, R><<<grid, PTHREADS, S::TOTAL, st>>>(mx, mw, p, bias, out, tiles, groups, work);
    B3D_LAUNCH_OK();
    b3d::add_variant("conv_tf32_persistent<%d,%d,%d,%d>", BN, STAGES, (int)WMN, R);
    return B3D_OK;
}

template <bool WMN>
int dispatch_persistent(int BN, int stack, const CUtensorMap& mx, const CUtensorMap& mw, const ConvParams& p, const float* bias,
                        float* out, int tiles, cudaStream_t st) {
    if (BN == 256) return launch_persistent<256, 4, WMN, 1>(mx, mw, p, bias, out, tiles, st);
    if (BN == 128) return stack ? launch_persistent<128, 4, WMN, 2>(mx, mw, p, bias, out, tiles, st) : launch_persistent<128, 3, WMN, 1>(mx, mw, p, bias, out, tiles, st);
    return stack ? launch_persistent<64, 3, WMN, 4>(mx, mw, p, bias, out, tiles, st) : launch_persistent<64, 4, WMN, 1>(mx, mw, p, bias, out, tiles, st);
}

int pow2_floor(int v) {
    int p = 1;
    while (p * 2 <= v) p *= 2;
    return p;
}

}  // namespace

extern "C" {

// x   [N, H, W, Cin]  NHWC fp32, Cin % 32 == 0
// wt  [ntaps, Cout, Cin] fp32 (tap-major, K-major rows)
// out [N, OH, OW, OC]; the tile grid covers (Hout, Wout) logical outputs, written to (osy*y+ooy, osx*x+oox)
int b3d_conv2d_tf32(const float* x, const float* wt, const float* bias, float* out, int N, int H, int W, int Cin,
                    int Hout, int Wout, int Cout, int ntaps, const int* dy, const int* dx, int sy, int sx, int OH,
                    int OW, int OC, int osy, int osx, int ooy, int oox, float leaky, int w_cin_major, const int* wtap,
                    int wtaps_total, double* stats, int fold_kh, int fold_pad, const b3d_conv_opts* opts, void* stream) {
    B3D_REQUIRE(N > 0 && H > 0 && W > 0 && Hout > 0 && Wout > 0 && Cout > 0, B3D_EINVAL, "b3d_conv2d_tf32: bad sizes");
    B3D_REQUIRE(Cin > 0 && Cin % BK == 0, B3D_EINVAL, "b3d_conv2d_tf32: Cin=%d must be a multiple of %d", Cin, BK);
    B3D_REQUIRE(ntaps >= 1 && ntaps <= MAX_TAPS && dy && dx, B3D_EINVAL, "b3d_conv2d_tf32: bad taps");
    B3D_REQUIRE(x && wt && out, B3D_EINVAL, "b3d_conv2d_tf32: null pointer");
    B3D_REQUIRE(sy >= 1 && sy <= 2 && sx >= 1 && sx <= 2, B3D_EINVAL, "b3d_conv2d_tf32: stride must be 1 or 2");
    if (!wtap) wtaps_total = ntaps;
    B3D_REQUIRE(wtaps_total >= ntaps || wtap, B3D_EINVAL, "b3d_conv2d_tf32: bad weight tap count");
    for (int t = 0; wtap && t < ntaps; ++t)
        B3D_REQUIRE(wtap[t] >= 0 && wtap[t] < wtaps_total, B3D_EINVAL, "b3d_conv2d_tf32: weight tap %d out of range", wtap[t]);
    B3D_CHECK_ALIGNED(x);
    B3D_CHECK_ALIGNED(wt);
    b3d::clear_variant();

    static const int persist_env = getenv("B3D_CONV_PERSIST") ? atoi(getenv("B3D_CONV_PERSIST")) : 1;
    const float* mask = opts ? opts->mask : nullptr;
    const float mslope = opts ? opts->mask_slope : 1.f;
    const int stats_sum = (opts && opts->stats_sum_only) ? 1 : 0;
    const int xpitch = (opts && opts->x_row_pitch) ? opts->x_row_pitch : W;
    // nclass > 1: the tap lists hold nclass groups of ntaps / nclass taps; class c writes at (class_ooy[c], class_oox[c])
    const int ncls = (opts && opts->nclass > 1) ? opts->nclass : 1;
    B3D_REQUIRE(ncls <= 4 && ntaps % ncls == 0 && (ncls == 1 || (sy == 1 && sx == 1 && fold_kh == 0)), B3D_EINVAL,
                "b3d_conv2d_tf32: nclass=%d needs <= 4 equal tap groups of a stride-1 launch", ncls);
    const int tpc = ntaps / ncls;                              // taps per class
    int cooy[4] = {ooy, ooy, ooy, ooy}, coox[4] = {oox, oox, oox, oox};
    for (int c = 0; c < ncls && ncls > 1; ++c) { cooy[c] = opts->class_ooy[c]; coox[c] = opts->class_oox[c]; }
    B3D_REQUIRE(xpitch >= W && (fold_kh == 0 || xpitch == W), B3D_EINVAL, "b3d_conv2d_tf32: x_row_pitch=%d must be >= W=%d (and absent with the on-the-fly fold)", xpitch, W);
    // statistics epilogue / on-the-fly fold / fused activation adjoint: persistent kernels
    const int persist = persist_env || stats != nullptr || fold_kh > 0 || mask != nullptr || ncls > 1;
    if (fold_kh > 0) {
        // x is the RAW stem input [N, H, W, 8]; the convolution is kh x kw with the kh rows folded into the K dimension:
        // Cin = 32 * ceil(8 kh / 32) "channels", taps = the kw horizontal ones (dy ignored), zero rows = the y padding
        B3D_REQUIRE(fold_kh <= 8 && Cin == 32 * ((8 * fold_kh + 31) / 32) && sy == 1 && sx == 1 && !w_cin_major && !wtap && Wout % BM == 0,
                    B3D_EINVAL, "b3d_conv2d_tf32: on-the-fly fold needs 8 input channels, stride 1 and Wout %% 128 == 0 (Wout=%d)", Wout);
    }
    // statistics are taken over every output pixel: a dense output, or the four parity classes of a stride-2 output
    const bool all_classes = ncls == 4 && osy == 2 && osx == 2;
    B3D_REQUIRE(!stats || mask || (osy == 1 && osx == 1) || all_classes, B3D_EINVAL, "b3d_conv2d_tf32: statistics need a dense output");
    static const int wide = getenv("B3D_CONV_BN256") ? atoi(getenv("B3D_CONV_BN256")) : 1;
    // 256-wide output-channel tiles halve the input-tile bytes per FLOP through the L2 -> SM fabric (the bound of the
    // per-tap formulation, profiles/r1_c_*.md) when there are >= 256 output channels and enough tiles to fill the GPU
    const bool bn256 = persist && wide && Cout % 256 == 0 && (long long)N * Hout * Wout / BM * (Cout / 256) * ncls >= 148;
    const int BN = bn256 ? 256 : Cout > 64 ? 128 : 64;
    cudaStream_t st = (cudaStream_t)stream;
    CUtensorMap mw;
    if (w_cin_major) {        // wt [ntaps, Cin, Cout]: the B operand is N-major (no weight transpose for dgrad)
        B3D_REQUIRE(Cout % 4 == 0, B3D_EINVAL, "b3d_conv2d_tf32: Cout=%d must be a multiple of 4 for cin-major weights", Cout);
        const uint64_t dims[3] = {(uint64_t)Cout, (uint64_t)Cin, (uint64_t)wtaps_total};
        const uint64_t strides[2] = {(uint64_t)Cout * 4, (uint64_t)Cout * Cin * 4};
        const uint32_t box[3] = {32, (uint32_t)BK, 1};
        if (int rc = tc::make_tmap_f32(&mw, wt, 3, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    } else {
        const uint64_t dims[3] = {(uint64_t)Cin, (uint64_t)Cout, (uint64_t)wtaps_total};
        const uint64_t strides[2] = {(uint64_t)Cin * 4, (uint64_t)Cout * Cin * 4};
        const uint32_t box[3] = {(uint32_t)BK, (uint32_t)BN, 1};
        if (int rc = tc::make_tmap_f32(&mw, wt, 3, dims, strides, box)) return rc;
    }

    // One launch covers output columns [xlo, xhi).  A width of "power of two + a few columns" (dgrad of an x-padded
    // input: 130, 66, 34 ...; stride-2 parity classes: 129, 65 ...) would leave a second, almost empty 128-pixel tile in
    // every row, so the remainder columns get a narrow strip launch of their own.
    // filter-grid detection for the row-window kernel (tc_conv3.cu): kh rows of kw horizontally consecutive taps; the weight
    // taps of a row form an arithmetic progression (identity, or the stride-2 dgrad parity classes' tap lists)
    int g_kw = 0, g_kh = 0, g_step = 0, g_wstep = 1;
    if (sy == 1 && sx == 1 && !w_cin_major && fold_kh == 0) {
        int kw_ = 1;
        while (kw_ < tpc && dy[kw_] == dy[0]) ++kw_;
        const int step = kw_ > 1 ? dx[1] - dx[0] : 1;
        const int wstep = (wtap && kw_ > 1) ? wtap[1] - wtap[0] : 1;
        bool grid_ok = tpc % kw_ == 0 && tpc / kw_ <= 5 && (kw_ == 2 || kw_ == 3 || kw_ == 5) && (step == 1 || step == -1) &&
                       wstep >= 1 && wstep <= 2 && (osy == osx) && (osy == 1 || osy == 2) && (ncls == 1 || wtap != nullptr);
        for (int t = 0; grid_ok && t < ntaps; ++t) {             // every class: the same column pattern, its own rows / weight taps
            const int tc_ = t % tpc, t0 = t - tc_;
            grid_ok = dy[t] == dy[t0 + (tc_ / kw_) * kw_] && dx[t] == dx[0] + (tc_ % kw_) * step;
            if (wtap) grid_ok = grid_ok && wtap[t] == wtap[t0 + (tc_ / kw_) * kw_] + (tc_ % kw_) * wstep;
        }
        static const int rowwin_env = getenv("B3D_CONV_ROWWIN") ? atoi(getenv("B3D_CONV_ROWWIN")) : 1;
        if (grid_ok && rowwin_env) { g_kw = kw_; g_kh = tpc / kw_; g_step = step; g_wstep = wstep; }
    }
    auto run = [&](int xlo, int xhi) -> int {
        const int wspan = xhi - xlo;
        if (g_kw && wspan >= BM) {
            b3d::RowWinArgs a{};
            a.x = x; a.wt = wt; a.bias = bias; a.out = out;
            a.N = N; a.H = H; a.W = W; a.Cin = Cin; a.Hout = Hout; a.Cout = Cout; a.xlo = xlo; a.xhi = xhi;
            a.kh = g_kh; a.kw = g_kw; a.ncls = ncls;
            a.dx0 = g_step > 0 ? dx[0] : dx[g_kw - 1];
            for (int t = 0; t < g_kw; ++t) a.shift[t] = dx[t] - a.dx0;
            a.OH = OH; a.OW = OW; a.OC = OC; a.leaky = leaky; a.stats = stats;
            a.osy = osy; a.osx = osx; a.wtaps_total = wtaps_total; a.wtap_step = g_wstep;
            a.mask = mask; a.mslope = mslope; a.stats_sum = stats_sum; a.xpitch = xpitch;
            for (int c = 0; c < ncls; ++c) {
                a.ooy[c] = cooy[c]; a.oox[c] = coox[c];
                for (int r = 0; r < g_kh; ++r) {
                    a.dy[c][r] = dy[c * tpc + r * g_kw];
                    a.wtap0[c][r] = wtap ? wtap[c * tpc + r * g_kw] : r * g_kw;
                }
            }
            const int rc = b3d::conv_rowwin_launch(a, st);
            if (rc <= 0) return rc;                           // launched (0) or a real error (< 0); 1 = not covered
        }
        ConvParams p{};
        p.N = N; p.Hout = Hout; p.Wout = xhi; p.Cout = Cout; p.xbase = xlo;
        p.BW = pow2_floor(wspan < BM ? wspan : BM);
        p.BH = pow2_floor(Hout < BM / p.BW ? Hout : BM / p.BW);
        p.BI = BM / (p.BW * p.BH);
        p.tiles_x = b3d::ceil_div(wspan, p.BW);
        p.tiles_y = b3d::ceil_div(Hout, p.BH);
        const int tiles = p.tiles_x * p.tiles_y * b3d::ceil_div(N, p.BI);
        p.ntaps = tpc; p.kslices = Cin / BK; p.sy = sy; p.sx = sx; p.ncls = ncls;
        for (int t = 0; t < ntaps; ++t) { p.dy[t] = dy[t]; p.dx[t] = dx[t]; p.wtap[t] = wtap ? wtap[t] : t; }
        for (int c = 0; c < 4; ++c) { p.cooy[c] = cooy[c]; p.coox[c] = coox[c]; }
        p.OH = OH; p.OW = OW; p.OC = OC; p.osy = osy; p.osx = osx; p.ooy = ooy; p.oox = oox;
        p.leaky = leaky;
        p.dbg_lbo = 4096; p.dbg_sbo = 512; p.dbg_lt = 1;     // 32-bit MN-major: SWIZZLE_128B_BASE32B, 4-row atoms
        p.stats = stats;
        p.mask = mask; p.mslope = mslope; p.stats_sum = stats_sum;
        p.fold = fold_kh; p.fold_y0 = -fold_pad;
        CUtensorMap mx;
        if (fold_kh > 0) {
            B3D_REQUIRE(p.BH == 1 && p.BI == 1, B3D_EINVAL, "b3d_conv2d_tf32: on-the-fly fold needs one-row tiles");
            const uint64_t dims[4] = {8, (uint64_t)W, (uint64_t)H, (uint64_t)N};                    // the raw NHWC tensor
            const uint64_t strides[3] = {32, (uint64_t)W * 32, (uint64_t)H * W * 32};
            const uint32_t box[4] = {8, (uint32_t)p.BW, 4, 1};                                     // 4 image rows per K slice
            if (int rc = tc::make_tmap_f32(&mx, x, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_32B)) return rc;
        } else {
        const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N};
        const uint64_t strides[3] = {(uint64_t)Cin * 4, (uint64_t)xpitch * Cin * 4, (uint64_t)H * xpitch * Cin * 4};
        const uint32_t box[4] = {(uint32_t)BK, (uint32_t)(sx * (p.BW - 1) + 1), (uint32_t)(sy * (p.BH - 1) + 1), (uint32_t)p.BI};
        const uint32_t es[4] = {1, (uint32_t)sx, (uint32_t)sy, 1};
        if (int rc = tc::make_tmap_f32(&mx, x, 4, dims, strides, box, es)) return rc;
        }
        // CTAs per SM x ring depth: short K loops (few taps x few channel slices) are dominated by pipeline fill, epilogue
        // and store drain, which only OTHER resident CTAs can hide -> more, shallower CTAs (profiles/r1_c_*.md)
        if (persist) {
            // stacked pixel tiles (1 CTA / SM, deeper stages) once there is work for ~2 waves of them
            static const int stack_env = getenv("B3D_CONV_STACK") ? atoi(getenv("B3D_CONV_STACK")) : 1;
            const int R = BN == 128 ? 2 : 4;
            const bool stack = stack_env && BN < 256 && (long long)b3d::ceil_div(tiles, R) * b3d::ceil_div(Cout, BN) * ncls >= 2 * 148;
            return w_cin_major ? dispatch_persistent<true>(BN, stack, mx, mw, p, bias, out, tiles, st)
                               : dispatch_persistent<false>(BN, stack, mx, mw, p, bias, out, tiles, st);
        }
        static const int occ_env = getenv("B3D_CONV_OCC") ? atoi(getenv("B3D_CONV_OCC")) : 0;
        const int occ = occ_env ? occ_env : 2;
        if (w_cin_major) {
            if (BN == 128) return occ >= 3 ? launch<128, 2, true, 3>(mx, mw, p, bias, out, tiles, st) : launch<128, 3, true, 2>(mx, mw, p, bias, out, tiles, st);
            return occ >= 4 ? launch<64, 2, true, 4>(mx, mw, p, bias, out, tiles, st)
                 : occ == 3 ? launch<64, 3, true, 3>(mx, mw, p, bias, out, tiles, st) : launch<64, 4, true, 2>(mx, mw, p, bias, out, tiles, st);
        }
        if (BN == 128) return occ >= 3 ? launch<128, 2, false, 3>(mx, mw, p, bias, out, tiles, st) : launch<128, 3, false, 2>(mx, mw, p, bias, out, tiles, st);
        return occ >= 4 ? launch<64, 2, false, 4>(mx, mw, p, bias, out, tiles, st)
             : occ == 3 ? launch<64, 3, false, 3>(mx, mw, p, bias, out, tiles, st) : launch<64, 4, false, 2>(mx, mw, p, bias, out, tiles, st);
    };
    const int bw_full = pow2_floor(Wout < BM ? Wout : BM);
    const int rem = Wout % bw_full;
    if (rem != 0 && rem * 8 <= bw_full && Wout > bw_full) {
        if (int rc = run(0, Wout - rem)) return rc;
        return run(Wout - rem, Wout);
    }
    return run(0, Wout);
}

// dy [N,Hout,Wout,Cout], x [N,H,W,Cin] NHWC (x already padded along x; Cin, Cout multiples of 4),
// dw [Cout,Cin,kh,kw] (accumulated into)
int b3d_conv2d_wgrad_tf32(const float* dy, const float* x, float* dw, int N, int H, int W, int Cin, int Hout, int Wout,
                          int Cout, int kh, int kw, int pad_y, int stride, int x_off, int tap_major, int fold_kh, int dy_row_pitch,
                          void* stream) {
    B3D_REQUIRE(N > 0 && Cin > 0 && Cout > 0 && H > 0 && W > 0 && Hout > 0 && Wout > 0, B3D_EINVAL,
                "b3d_conv2d_wgrad_tf32: bad sizes");
    // x_off < 0 reads columns left of x as zeros (the TMA fills out-of-bounds boxes): the up-convolution's weight gradient
    B3D_REQUIRE(kh * kw <= MAX_TAPS && (stride == 1 || stride == 2) && x_off > -kw, B3D_EINVAL, "b3d_conv2d_wgrad_tf32: bad kernel/stride");
    B3D_REQUIRE(dy && x && dw, B3D_EINVAL, "b3d_conv2d_wgrad_tf32: null pointer");
    B3D_REQUIRE(Cin % 32 == 0 && Cout % 32 == 0, B3D_EINVAL,
                "b3d_conv2d_wgrad_tf32: Cin=%d and Cout=%d must be multiples of 32 (pad the channels with zeros)", Cin, Cout);
    B3D_CHECK_ALIGNED(dy);
    B3D_CHECK_ALIGNED(x);
    b3d::clear_variant();
    WgradParams p{};
    p.N = N; p.Hout = Hout; p.Wout = Wout; p.Cout = Cout; p.Cin = Cin;
    p.BWk = pow2_floor(Wout < BK ? Wout : BK);
    p.BHk = BK / p.BWk;
    p.kx = b3d::ceil_div(Wout, p.BWk);
    p.ky = b3d::ceil_div(Hout, p.BHk);
    p.kh = kh; p.kw = kw; p.pad_y = pad_y; p.st = stride; p.xoff = x_off; p.tapmajor = tap_major ? 1 : 0;
    p.fold = fold_kh;
    B3D_REQUIRE(fold_kh == 0, B3D_EINVAL,
                "b3d_conv2d_wgrad_tf32: the on-the-fly fold is not available for the weight gradient (TMA pads 32-byte inner boxes "
                "to 128-byte lines under the 128B swizzles the MN-major tf32 operand needs): pass the materialised fold");
    if (tap_major) B3D_CHECK_ALIGNED(dw);
    // a row of kw taps per CTA when the K slice is a 32-pixel row segment (Wout >= 32) of a stride-1 conv
    int T = 1;
    p.tstep = 1;
    if (Wout >= BK && !getenv("B3D_WGRAD_T1")) {
        if (stride == 1 && (kw == 3 || kw == 5)) T = kw;
        if (stride == 2 && kw == 4) { T = 2; p.tstep = 2; }      // taps {0,2} and {1,3}: rows t of one strided window
    }
    const int BN = (Cin > 64 && T != 5) ? 128 : 64;          // T * BN <= 512 TMEM columns
    const int base_ctas = b3d::ceil_div(Cout, BM) * b3d::ceil_div(Cin, BN) * kh * (kw / T);
    const long long ktotal = (long long)N * p.kx * p.ky;
    int splits = ((T == 2 ? 4 : 2) * 148 + base_ctas - 1) / base_ctas;   // ~2 waves of CTAs per resident CTA slot
    if (splits > ktotal / 8) splits = (int)(ktotal / 8);         // at least 8 K slices per CTA
    if (splits < 1) splits = 1;
    p.splits = splits;

    CUtensorMap mdy, mx;
    {   // dims: (32 channels, W, H, N, channel block) — the block dim is outermost so that a box of BM/32 blocks is contiguous
        const uint64_t dims[5] = {32, (uint64_t)Wout, (uint64_t)Hout, (uint64_t)N, (uint64_t)Cout / 32};
        const uint64_t dpitch = dy_row_pitch > 0 ? dy_row_pitch : Wout;            // pixels per row of dy in memory
        B3D_REQUIRE(dpitch >= (uint64_t)Wout, B3D_EINVAL, "b3d_conv2d_wgrad_tf32: dy_row_pitch=%d must be >= Wout=%d", dy_row_pitch, Wout);
        const uint64_t strides[4] = {(uint64_t)Cout * 4, dpitch * Cout * 4, (uint64_t)Hout * dpitch * Cout * 4, 128};
        const uint32_t box[5] = {32, (uint32_t)p.BWk, (uint32_t)p.BHk, 1, (uint32_t)(BM / 32)};
        if (int rc = tc::make_tmap_f32(&mdy, dy, 5, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    }
    if (fold_kh > 0) {
        const uint64_t dims[4] = {8, (uint64_t)H, (uint64_t)W, (uint64_t)N};                        // (c, row, x, n)
        const uint64_t strides[3] = {(uint64_t)W * 32, 32, (uint64_t)H * W * 32};
        const uint32_t box[4] = {8, 4, (uint32_t)(T == 1 ? p.BWk : 36), 1};
        if (int rc = tc::make_tmap_f32(&mx, x, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    } else {
        const uint64_t dims[5] = {32, (uint64_t)W, (uint64_t)H, (uint64_t)N, (uint64_t)Cin / 32};
        const uint64_t strides[4] = {(uint64_t)Cin * 4, (uint64_t)W * Cin * 4, (uint64_t)H * W * Cin * 4, 128};
        const uint32_t box[5] = {32, (uint32_t)(T == 1 ? stride * (p.BWk - 1) + 1 : stride * 35 + 1), (uint32_t)(stride * (p.BHk - 1) + 1), 1,
                                 (uint32_t)(BN / 32)};
        const uint32_t es[5] = {1, (uint32_t)stride, (uint32_t)stride, 1, 1};
        if (int rc = tc::make_tmap_f32(&mx, x, 5, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
    }
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(b3d::ceil_div(Cout, BM), b3d::ceil_div(Cin, BN), kh * (kw / T) * splits);
    const bool two = !getenv("B3D_WGRAD_1CTA");           // two CTAs per SM (half-depth ring) where TMEM has room for both
    if (T == 2 && BN == 128) return two ? launch_wgrad<128, 3, 2>(mdy, mx, p, dw, grid, st) : launch_wgrad<128, 6, 2>(mdy, mx, p, dw, grid, st);
    if (T == 2) return two ? launch_wgrad<64, 4, 2>(mdy, mx, p, dw, grid, st) : launch_wgrad<64, 8, 2>(mdy, mx, p, dw, grid, st);
    if (T == 3 && BN == 128) return launch_wgrad<128, 6, 3>(mdy, mx, p, dw, grid, st);
    // Cout = Cin = 64 rows of three taps: nothing is saturated with one CTA per SM (ncu: tensor pipe 35 %, L2 14 %): two
    // half-depth CTAs per SM overlap each other's TMA latency and epilogue (B3D_WGRAD_T3=1 restores the deep single ring)
    static const int t3_one = getenv("B3D_WGRAD_T3") ? atoi(getenv("B3D_WGRAD_T3")) : 0;
    if (T == 3) return t3_one ? launch_wgrad<64, 8, 3>(mdy, mx, p, dw, grid, st) : launch_wgrad<64, 4, 3>(mdy, mx, p, dw, grid, st);
    if (T == 5) return launch_wgrad<64, 8, 5>(mdy, mx, p, dw, grid, st);
    // single taps: the deep single-CTA ring measured faster (profiles/r1_conv_layers.md)
    if (BN == 128) return launch_wgrad<128, 6, 1>(mdy, mx, p, dw, grid, st);
    return launch_wgrad<64, 8, 1>(mdy, mx, p, dw, grid, st);
}

}  // extern "C"
