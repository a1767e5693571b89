// Fused tcgen05 pipeline for chains of Bayesian layers on small feature maps.
//
// Between fused layers the activation lives in HBM "tiled packed": [B/128][F/64][planes] blocks of
// 128 rows x 128 B (64 bf16 of the NHWC-flattened (pixel, channel) axis), each block already in the
// SWIZZLE_128B shared-memory image, written that way by the producing epilogue; for LRT consumers the
// element-wise square is interleaved behind every x block -- so an A (A^2) tile is ONE 16 KB cp.async.bulk
// and x^2 never has to be recomputed.
//
//  (P) tap_prep_kernel / tap_prep_conv_kernel : like weight_prep_kernel but tap-major:
//      [tap][cout block][cin block][plane][NG x 64] bf16 sub-tiles, pre-swizzled, + one zero sub-tile.
//      softplus / eps / KL exactly once per weight.
//
//  (G) tap_gemm_kernel : "conv on a small map == block-structured dense layer".
//      Rows = 128 images, K walks (input pixel, 64-channel block), each output
//      column group = (output pixel, NG output channels).  For every K step the
//      tap that links the group's output pixel to the input pixel is computed; if
//      it falls outside the kernel window the MMA (and the weight copy) is skipped
//      -- zero padding costs nothing (AlexNet conv3-5: 4 of 9 taps are live).
//        warps 9-12 : producers (each owns ring stages): cp.async.bulk of A / A^2 blocks and of the
//                     live weight sub-tiles, mbarrier complete_tx
//        warp 8     : tcgen05.mma issuer (M=128, N=64, bf16 -> fp32 TMEM; LRT: 2nd accumulator)
//        warps 0-7  : LRT noise tile (Philox) during the main loop, then the epilogue -- tcgen05.ld,
//                     bias, sqrt(var)*eps, 2x2 max-pool across the four column groups, activation,
//                     tiled-packed bf16 (+square) or fp32 store
#pragma once
#include "fwd_tc.cuh"

namespace bbb {


struct FusedArgs {
    Geom g;
    int variant, sample, has_bias, act, kl_convention;
    float prior_mu, prior_sigma;
    const float *w_mu, *w_rho, *b_mu, *b_rho, *eps_a, *eps_b;
    NoiseKey key; const unsigned long long* stream_base;
    double* kl_partials; unsigned int* kl_counter; float* kl_out;
    __nv_bfloat16* wtiles; float* bias_ws;
    int planes, ng, n_cblk, n_kblk, taps;
    int prev_hw;                 // linear fed by a flattened HxW map: k' = pix*C + c  <->  ref k = c*HW + pix
    const void* x; const void* x_sq;   // tiled packed input (and its square)
    void* y; void* y_sq;
    int out_mode, out_pitch, pool, in_pitch;   // pitches = F (columns) of the tiled packed matrices
    long long* trace;            // debug: per-CTA clock64 checkpoints (nullptr in production)
    long long* tl_prep; long long* tl_gemm;   // debug: timeline slots of the two launches (nullptr in production)
    int units;                   // K blocks per pipeline step (TAP_UNITS, or 1 in the two-CTAs-per-SM LRT configuration)
    McFold fold;                 // MC samples folded into the batch (rows = 0: off)
};

__host__ __device__ inline size_t fused_wtile_elems(const FusedArgs& a) { return (size_t)a.planes * a.ng * 64; }
inline size_t fused_workspace_bytes(const Geom& g) {
    // worst case NG=16 padding of Cout, 2 planes
    const size_t cpad = (size_t)(g.N + 63) / 64 * 64, kpad = (size_t)(g.Cin + 63) / 64 * 64;
    return cpad * kpad * g.KHW * 2 * 2 + 32768 /* zero sub-tile (<= 2 planes x 128 rows x 128 B) */ + 2 * cpad * 4;
}

// ------------------------------------------------------------- (P) tap prep
template <int VARIANT>
__global__ void __launch_bounds__(256)
tap_prep_kernel(const FusedArgs p) {
    __shared__ double red[32];
    constexpr bool LRT = VARIANT == BBB_VARIANT_LRT;
    const Geom& g = p.g;
    const NoiseKey nkey = effective_key(p.key, p.stream_base);
    const bool stoch = p.sample != 0, do_kl = p.kl_out != nullptr;
    const int cprev = g.Cin / p.prev_hw;
    const size_t sub = fused_wtile_elems(p);
    const int per_sub = p.ng * 8;                                  // (row, 8-wide K chunk) items per sub-tile
    const long n_items = (long)p.taps * p.n_cblk * p.n_kblk * per_sub;
    double kl_acc = 0.0;
    tl_enter(p.tl_prep);
    for (long gi = (long)blockIdx.x * blockDim.x + threadIdx.x; gi < n_items; gi += (long)gridDim.x * blockDim.x) {
        const int st = (int)(gi / per_sub), item = (int)(gi - (long)st * per_sub);
        const int kb = st % p.n_kblk, cb = (st / p.n_kblk) % p.n_cblk, tap = st / (p.n_kblk * p.n_cblk);
        __nv_bfloat16* dst = p.wtiles + (size_t)st * sub;          // st == (tap*n_cblk + cb)*n_kblk + kb
        const int row = item % p.ng, chunk = item / p.ng;
        const int n = cb * p.ng + row;
        float w[8], s2[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int kq = kb * 64 + chunk * 8 + e;                // packed input-channel index
            float wv = 0.0f, sv = 0.0f;
            if (n < g.N && kq < g.Cin) {
                const int cin = (p.prev_hw > 1) ? ((kq % cprev) * p.prev_hw + kq / cprev) : kq;
                const size_t wi = (size_t)n * g.K + (size_t)cin * g.KHW + tap;
                const float mu = __ldg(p.w_mu + wi);
                float sigma = 0.0f;
                if (stoch || do_kl) sigma = softplus_sigma_fast(__ldg(p.w_rho + wi));
                if (LRT) { wv = mu; sv = sigma * sigma; }
                else if (stoch) {
                    const float e_ = p.eps_a ? __ldg(p.eps_a + wi) : normal1(wi, nkey);
                    wv = mu + e_ * sigma;
                } else wv = mu;
                if (do_kl) kl_acc += (double)kl_term_fast(mu, sigma, p.prior_mu, p.prior_sigma, p.kl_convention);
            }
            w[e] = wv; s2[e] = sv;
        }
        // K-major SWIZZLE_128B image: row r = 128 contiguous bytes, its 16-byte chunk c stored at chunk (c ^ (r & 7))
        const int sw = row * 64 + ((chunk ^ (row & 7)) << 3);
        const uint4 o = make_uint4(pack_bf16(w[0], w[1]), pack_bf16(w[2], w[3]), pack_bf16(w[4], w[5]), pack_bf16(w[6], w[7]));
        *reinterpret_cast<uint4*>(dst + sw) = o;
        if (p.planes == 2) {
            const uint4 o2 = make_uint4(pack_bf16(s2[0], s2[1]), pack_bf16(s2[2], s2[3]), pack_bf16(s2[4], s2[5]), pack_bf16(s2[6], s2[7]));
            *reinterpret_cast<uint4*>(dst + p.ng * 64 + sw) = o2;
        }
    }
    // one all-zero sub-tile behind the real ones: staged for pool-window pixels whose tap is outside the kernel
    for (long gi = (long)blockIdx.x * blockDim.x + threadIdx.x; gi < (long)(sub / 8); gi += (long)gridDim.x * blockDim.x)
        reinterpret_cast<uint4*>(p.wtiles + (size_t)p.taps * p.n_cblk * p.n_kblk * sub)[gi] = make_uint4(0u, 0u, 0u, 0u);
    {   // bias: prepared (and its KL counted) by the first CTAs, one thread per channel
        const int npad = p.n_cblk * p.ng;
        for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < npad; n += gridDim.x * blockDim.x) {
            float bm = 0.0f, bv = 0.0f;
            if (p.has_bias && n < g.N) {
                const float mu = __ldg(p.b_mu + n);
                const float sigma = (stoch || do_kl) ? softplus_sigma_fast(__ldg(p.b_rho + n)) : 0.0f;
                if (LRT) { bm = mu; bv = sigma * sigma; }
                else if (stoch) {
                    const float e_ = p.eps_b ? __ldg(p.eps_b + n) : normal1((uint64_t)g.N * g.K + n, nkey);
                    bm = mu + e_ * sigma;
                } else bm = mu;
                if (do_kl) kl_acc += (double)kl_term_fast(mu, sigma, p.prior_mu, p.prior_sigma, p.kl_convention);
            }
            p.bias_ws[n] = bm;
            p.bias_ws[npad + n] = bv;
        }
    }
    if (do_kl) {
        const double tot = block_sum(kl_acc, red);
        if (threadIdx.x == 0) kl_publish(tot, blockIdx.x, gridDim.x, p.kl_partials, p.kl_counter, p.kl_out);
    }
    tl_exit(p.tl_prep);
}

// ------------------------------------------------- (P2) tap prep, conv layers
// Same outputs as tap_prep_kernel for layers with a real kernel window (KHW > 1, prev_hw == 1), but reading the
// parameters the way they lie in memory.  tap_prep_kernel's work item is one 16-byte output chunk = 8 input
// channels of ONE tap, i.e. eight 4-byte loads KHW floats apart per thread and a different row per lane: every
// warp load touches 32 lines and every 32-byte sector is fetched KHW times (by KHW different CTAs).  That made the
// preps LSU-bound (17-32 us per AlexNet layer for 0.3-0.9 M weights) and they share the machine with the first
// GEMMs.  Here a CTA owns R output channels x one 64-input-channel block: each row's 64*KHW floats are contiguous
// in OIHW order and are read with consecutive lanes on consecutive floats; softplus / eps / KL are element-wise, so
// they are applied right there; the bf16 results go through shared memory ([plane][tap][row][cin]) and leave as the
// same pre-swizzled 16-byte chunks, 1 KB contiguous per (tap, plane).
constexpr int PREP2_BATCH = 4;                                     // loads in flight per thread
__host__ __device__ inline int prep2_slab(int R) { return R * 64 + 8; }   // bf16 per (plane, tap) slab; +8 keeps 16 B alignment, skews banks

template <int VARIANT>
__global__ void __launch_bounds__(256)
tap_prep_conv_kernel(const FusedArgs p, const int R) {
    extern __shared__ __align__(16) uint8_t prep2_smem[];
    __shared__ double red[32];
    constexpr bool LRT = VARIANT == BBB_VARIANT_LRT;
    __nv_bfloat16* sm = reinterpret_cast<__nv_bfloat16*>(prep2_smem);
    const Geom& g = p.g;
    const NoiseKey nkey = effective_key(p.key, p.stream_base);
    const bool stoch = p.sample != 0, do_kl = p.kl_out != nullptr;
    const int KHW = g.KHW, L = 64 * KHW, PS = prep2_slab(R);
    const size_t sub = fused_wtile_elems(p);
    const int n_units = (p.n_cblk * p.ng / R) * p.n_kblk;
    const int dc = 256 / KHW, dq = 256 - dc * KHW;                  // (cin, tap) advance of a 256-element stride
    double kl_acc = 0.0;
    tl_enter(p.tl_prep);
    for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
        const int rb = unit / p.n_kblk, kb = unit - rb * p.n_kblk;
        const int n0 = rb * R, cin0 = kb * 64;
        const int total = R * L;
        // ---- phase 1: coalesced loads, element-wise math, bf16 into smem ----
        int cin = threadIdx.x / KHW, tap = threadIdx.x - cin * KHW, r = 0;
        while (cin >= 64) { cin -= 64; ++r; }
        for (int e0 = threadIdx.x; e0 < total; e0 += 256 * PREP2_BATCH) {
            float mu[PREP2_BATCH], rho[PREP2_BATCH];
            size_t wi[PREP2_BATCH];
            int so[PREP2_BATCH];                                    // smem offset of the element, -1: past the end
            bool ok[PREP2_BATCH];
#pragma unroll
            for (int u = 0; u < PREP2_BATCH; ++u) {
                const bool in = e0 + 256 * u < total;
                const int n = n0 + r;
                ok[u] = in && n < g.N && cin0 + cin < g.Cin;
                wi[u] = (size_t)n * g.K + (size_t)(cin0 + cin) * KHW + tap;
                so[u] = in ? tap * PS + r * 64 + cin : -1;
                mu[u] = ok[u] ? __ldg(p.w_mu + wi[u]) : 0.0f;
                rho[u] = (ok[u] && (stoch || do_kl)) ? __ldg(p.w_rho + wi[u]) : 0.0f;
                tap += dq; cin += dc;
                if (tap >= KHW) { tap -= KHW; ++cin; }
                while (cin >= 64) { cin -= 64; ++r; }
            }
#pragma unroll
            for (int u = 0; u < PREP2_BATCH; ++u) {
                if (so[u] < 0) continue;
                float wv = 0.0f, sv = 0.0f;
                if (ok[u]) {
                    const float sigma = (stoch || do_kl) ? softplus_sigma_fast(rho[u]) : 0.0f;
                    if (LRT) { wv = mu[u]; sv = sigma * sigma; }
                    else if (stoch) {
                        const float e_ = p.eps_a ? __ldg(p.eps_a + wi[u]) : normal1(wi[u], nkey);
                        wv = mu[u] + e_ * sigma;
                    } else wv = mu[u];
                    if (do_kl) kl_acc += (double)kl_term_fast(mu[u], sigma, p.prior_mu, p.prior_sigma, p.kl_convention);
                }
                sm[so[u]] = __float2bfloat16_rn(wv);
                if (p.planes == 2) sm[KHW * PS + so[u]] = __float2bfloat16_rn(sv);
            }
        }
        __syncthreads();
        // ---- phase 2: 16-byte chunks (8 input channels of one tap) out, in the SW128 image order ----
        const int items = p.planes * KHW * R * 8;
        for (int it = threadIdx.x; it < items; it += 256) {
            const int chunk = it & 7, rr = (it >> 3) % R, pt = it / (8 * R);      // pt = plane*KHW + tap
            const int plane = pt / KHW, tp = pt - plane * KHW;
            const uint4 v = *reinterpret_cast<const uint4*>(sm + (size_t)pt * PS + rr * 64 + chunk * 8);
            const int n = n0 + rr, cb = n / p.ng, row = n - cb * p.ng;
            const size_t st = ((size_t)tp * p.n_cblk + cb) * p.n_kblk + kb;
            __nv_bfloat16* dst = p.wtiles + st * sub + (size_t)plane * p.ng * 64 + row * 64 + ((chunk ^ (row & 7)) << 3);
            *reinterpret_cast<uint4*>(dst) = v;
        }
        __syncthreads();
    }
    // one all-zero sub-tile behind the real ones: staged for pool-window pixels whose tap is outside the kernel
    for (long gi = (long)blockIdx.x * blockDim.x + threadIdx.x; gi < (long)(sub / 8); gi += (long)gridDim.x * blockDim.x)
        reinterpret_cast<uint4*>(p.wtiles + (size_t)p.taps * p.n_cblk * p.n_kblk * sub)[gi] = make_uint4(0u, 0u, 0u, 0u);
    {   // bias: prepared (and its KL counted) by the first CTAs, one thread per channel
        const int npad = p.n_cblk * p.ng;
        for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < npad; n += gridDim.x * blockDim.x) {
            float bm = 0.0f, bv = 0.0f;
            if (p.has_bias && n < g.N) {
                const float mu = __ldg(p.b_mu + n);
                const float sigma = (stoch || do_kl) ? softplus_sigma_fast(__ldg(p.b_rho + n)) : 0.0f;
                if (LRT) { bm = mu; bv = sigma * sigma; }
                else if (stoch) {
                    const float e_ = p.eps_b ? __ldg(p.eps_b + n) : normal1((uint64_t)g.N * g.K + n, nkey);
                    bm = mu + e_ * sigma;
                } else bm = mu;
                if (do_kl) kl_acc += (double)kl_term_fast(mu, sigma, p.prior_mu, p.prior_sigma, p.kl_convention);
            }
            p.bias_ws[n] = bm;
            p.bias_ws[npad + n] = bv;
        }
    }
    if (do_kl) {
        const double tot = block_sum(kl_acc, red);
        if (threadIdx.x == 0) kl_publish(tot, blockIdx.x, gridDim.x, p.kl_partials, p.kl_counter, p.kl_out);
    }
    tl_exit(p.tl_prep);
}

// ------------------------------------------------------------- UMMA helpers
// two packed bf16 -> their squares (exact product, one rounding: same value as bf16(float(x) * float(x)))
__device__ __forceinline__ uint32_t bf16x2_sq(uint32_t v) {
    __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&v);
    h = __hmul2(h, h);
    return *reinterpret_cast<uint32_t*>(&h);
}
// K-major SWIZZLE_128B descriptor: 8-row groups 1024 B apart, layout_type = 2 at [61,64)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
           (1ull << 46) | (2ull << 61);
}

constexpr int TAP_MAX_ITEMS = 64;       // live (input pixel, 64-channel block) pairs per tile (control block must stay < 2 KB)
constexpr int TAP_UNITS = 2;            // K blocks handled per pipeline step (one mbarrier phase)
static_assert(true, "");
struct FusedSmem {
    unsigned long long full[4], empty[4], accum;
    uint32_t tmem_base, n_items;
    float bias[128], bvar[128];     // this tile's output columns (BN <= 128)
    // K-loop schedule, built once per CTA: x = ipix | kb << 16, y = the four column groups' taps (0xFF = outside the
    // kernel window -> zero sub-tile).  A pipeline step covers TAP_UNITS consecutive items: the fixed cost of a stage
    // hand-off (~500-900 cycles measured: barrier round trip + TMA issue + first-MMA start-up) is paid per STEP.
    int2 items[TAP_MAX_ITEMS];
    int taps_px[64];                // per input pixel: packed taps (staging for the schedule build)
};

// tap linking output pixel (oh,ow) with input pixel (ih,iw); -1 if outside the kernel window
__device__ __forceinline__ int tap_of(const Geom& g, int oh, int ow, int ih, int iw) {
    const int r = ih - oh * g.SH + g.PH, s = iw - ow * g.SW + g.PW;
    if ((unsigned)r < (unsigned)g.KH && (unsigned)s < (unsigned)g.KW) return r * g.KW + s;
    return -1;
}

__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
    uint32_t r0, r1, r2, r3;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
}

// LRT activation noise of image b, output pixel pix, channels [n, n+4): Philox element index is
// the NHWC-flat index ((b*OHW + pix)*N + n), so four consecutive channels share one Philox call.
__device__ __forceinline__ float4 act_noise4(const NoiseKey& k, int b, int pix, int n, int OHW, int N) {
    const uint64_t o = ((uint64_t)b * OHW + pix) * N + n;
    if ((N & 3) == 0) return normal4(o >> 2, k);
    float4 z;
    z.x = normal1(o, k); z.y = normal1(o + 1, k); z.z = normal1(o + 2, k); z.w = normal1(o + 3, k);
    return z;
}

// Thread roles (416 threads): warps 0-7 epilogue (two groups of four; group h owns half of the tile's 64
// columns; warps w and w+4 read the same TMEM lanes), warp 8 MMA issuer, warps 9-12 TMA producers (one
// elected thread each; the copies of a stage are dealt round-robin so their ~100-cycle issue costs overlap).
constexpr int TAP_THREADS = 416, TAP_NPROD = 4;

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
                   "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// TMEM columns of a tile (BN = tile width, 64 or 128): [0,BN) mean accumulator, [BN,2BN) variance accumulator (LRT),
// [2BN,3BN) the tile's LRT noise.  The noise tile is drawn (Philox) by the epilogue warps WHILE the main loop runs and
// parked in tensor memory: no shared memory, no registers held across the main loop, and the epilogue stays a short rolled
// loop with static register indices (a 64-value register array would force full unrolling; straight-line code that runs
// once per CTA is what the cold instruction cache punishes -- DESIGN.md 5).
//
// BN: every SS-mode tcgen05.mma pulls (128 + BN) * 32 B of operands out of shared memory at 64 B/clk (measured, DESIGN.md
// 5), i.e. 96 cycles for the 32 cycles of math of an N=64 MMA, 128 for the 64 cycles of an N=128 one: the wider tile
// raises the tensor-pipe ceiling from 1/3 to 1/2 and is used whenever it still leaves enough CTAs for the machine.
// MINB = resident CTAs per SM the register allocation is sized for (1: configuration A, 2: configuration B)
template <int MINB, int BN>
__global__ void __launch_bounds__(TAP_THREADS, MINB)
tap_gemm_kernel(const FusedArgs p, const int stages) {
    extern __shared__ uint8_t smem_raw[];
    constexpr uint32_t TB = BN * 128;                   // bytes of one B plane of a K block (BN rows x 64 bf16)
    const Geom& g = p.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int planes = p.planes;
    const bool two = planes == 2;
    const int ng = p.ng, groups = BN / ng;

    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* sm = smem_raw + (base - raw);
    FusedSmem* ctl = reinterpret_cast<FusedSmem*>(sm);
    const uint32_t tiles_off = 2048u;
    const uint32_t unit_bytes = (uint32_t)planes * (TC_A_BYTES + TB);   // one K block: [A][A^2][B planes]
    const int units = p.units;
    const uint32_t stage_bytes = (uint32_t)units * unit_bytes;
    const uint32_t a2_off = TC_A_BYTES, b_off = (uint32_t)planes * TC_A_BYTES;

    // output tile -> (pixel set, cout block)
    const int n_tile = blockIdx.x, m0 = blockIdx.y * TC_BM;
    const int cb = n_tile % p.n_cblk, pset = n_tile / p.n_cblk;
    // pixel of column group q: pool -> the q-th pixel of the 2x2 window `pset`; otherwise the single pixel `pset`
    const int win_y = p.pool ? pset / (g.OW >> 1) : 0, win_x = p.pool ? pset - win_y * (g.OW >> 1) : 0;
    auto group_pix = [&](int q, int& oh, int& ow) {
        if (p.pool) { oh = 2 * win_y + (q >> 1); ow = 2 * win_x + (q & 1); }
        else { oh = pset / g.OW; ow = pset - oh * g.OW; }
    };

    // debug trace: 128 slots per CTA -- [0,8) phase checkpoints, [8,40) MMA thread: full[s] passed at step it,
    // [48,88) producer 0: empty[s] passed at step it, [88,128) producer 0: step it issued
    long long* tr = p.trace ? p.trace + (size_t)(blockIdx.y * gridDim.x + blockIdx.x) * 128 : nullptr;
    if (tr && threadIdx.x == 0) tr[0] = clock64();
    tl_enter(p.tl_gemm);
    pdl_trigger();
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(smem_u32(&ctl->full[s]), 1);
            mbar_init(smem_u32(&ctl->empty[s]), 1);
        }
        mbar_init(smem_u32(&ctl->accum), 1);
        fence_barrier_init();
    }
    // K-loop schedule: one thread per input pixel works out the taps (integer divisions), thread 64 compacts
    if (threadIdx.x >= 128 && threadIdx.x < 128 + g.HW) {
        const int ipix = threadIdx.x - 128;
        const int ih = ipix / g.W, iw = ipix - ih * g.W;
        uint32_t taps = 0;
        for (int q = 0; q < 4; ++q) {
            int oh, ow;
            group_pix(q, oh, ow);
            const int tp = (q < groups) ? tap_of(g, oh, ow, ih, iw) : -1;
            taps |= (uint32_t)(tp >= 0 ? tp : 0xFF) << (8 * q);
        }
        ctl->taps_px[ipix] = (int)taps;
    }
    __syncthreads();
    if (threadIdx.x == 64) {
        int n = 0;
        for (int ipix = 0; ipix < g.HW; ++ipix) {
            const int taps = ctl->taps_px[ipix];
            if ((uint32_t)taps == 0xFFFFFFFFu) continue;
            for (int kb = 0; kb < p.n_kblk; ++kb) ctl->items[n++] = make_int2(ipix | (kb << 16), taps);
        }
        ctl->n_items = (uint32_t)n;
    }
    const bool philox = two && !p.eps_a;
    const uint32_t tmem_cols = philox ? 4u * BN : (two ? 2u * BN : (uint32_t)BN);     // power of two >= 3 BN when the noise tile lives there
    constexpr uint32_t NOISE_COL = 2u * BN;
    if (warp == 8) tmem_alloc(smem_u32(&ctl->tmem_base), tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = ctl->tmem_base;
    if (tr && threadIdx.x == 0) tr[1] = clock64();

    const int n_items = (int)ctl->n_items;
    const int n_steps = (n_items + units - 1) / units;

    if (warp >= 9) {
        // ======================= TMA producers ==================================
        // The WHOLE warp executes the loop and the mbarrier waits; only the copies are issued by one lane.
        // (tools/pipe_probe.cu: a try_wait that blocks with a single active lane is woken ~750 cycles late --
        //  apparently by a time-out poll -- while a fully converged warp is woken as soon as the phase flips.)
        // Issuing a stage costs one thread several hundred cycles of dependent latency (tools/tma_probe.cu: ~350
        // cycles per expect_tx + cp.async.bulk pair) while the data lands ~250 cycles later, so the STEPS are dealt
        // round-robin to the four producer warps: four issue chains run concurrently.
        // A producer must see EVERY phase of the stage it fills (parity waits alias after two phases), so at most
        // `stages` producers take part and producer p owns stage p (mod nprod).
        const int pid = warp - 9;
        const int nprod = min(TAP_NPROD, stages);
        pdl_wait();                                      // A / A^2 are the previous layer's output
        tl_dep(p.tl_gemm, 288);
        const size_t sub_elems = (size_t)planes * ng * 64;
        const __nv_bfloat16* zero_tile = p.wtiles + (size_t)p.taps * p.n_cblk * p.n_kblk * sub_elems;
        const uint32_t gbytes = (uint32_t)ng * 128;                     // one group, one plane
        const uint32_t a_copy = (uint32_t)planes * TC_A_BYTES;
        const uint32_t unit_tx = a_copy + (uint32_t)(groups * planes) * gbytes;
        const size_t a_row0 = (size_t)blockIdx.y * (p.in_pitch >> 6);   // first 16 KB block of this row tile
#pragma unroll 1
        for (int it = pid; it < n_steps && pid < nprod; it += nprod) {
            const int s = it % stages;
            __syncwarp();
            mbar_wait(smem_u32(&ctl->empty[s]), ((uint32_t)(it / stages) & 1u) ^ 1u);
            if (tr && it < 40 && lane == 0) tr[48 + it] = clock64();
            if (lane == 0) {
                const int i0 = it * units, nu = min(units, n_items - i0);
                const uint32_t bar = smem_u32(&ctl->full[s]);
                mbar_arrive_expect_tx(bar, unit_tx * nu);
#pragma unroll 1
                for (int u = 0; u < nu; ++u) {
                    const int2 item = ctl->items[i0 + u];
                    const int ipix = item.x & 0xffff, kb = item.x >> 16;
                    const uint32_t st = base + tiles_off + (uint32_t)s * stage_bytes + (uint32_t)u * unit_bytes;
                    // x and x^2 blocks are interleaved in global memory and adjacent in the stage: one copy
                    const size_t a_blk = (a_row0 + (size_t)ipix * p.n_kblk + kb) * (size_t)(planes * 128 * 64);
                    bulk_g2s(st, reinterpret_cast<const __nv_bfloat16*>(p.x) + a_blk, a_copy, bar);
                    // weight planes: [plane][group][ng rows x 128 B] -> every plane is one BN-row SW128 tile
#pragma unroll 1
                    for (int q = 0; q < groups; ++q) {
                        const int tp = (item.y >> (8 * q)) & 0xFF;
                        const __nv_bfloat16* sp = tp != 0xFF ? p.wtiles + ((size_t)(tp * p.n_cblk + cb) * p.n_kblk + kb) * sub_elems : zero_tile;
                        if (groups == 1) {           // [mu | sigma^2] of the sub-tile are contiguous here and in the stage
                            bulk_g2s(st + b_off, sp, (uint32_t)planes * gbytes, bar);
                        } else {
                            bulk_g2s(st + b_off + q * gbytes, sp, gbytes, bar);
                            if (two) bulk_g2s(st + b_off + TB + q * gbytes, tp != 0xFF ? sp + ng * 64 : zero_tile, gbytes, bar);
                        }
                    }
                }
                if (tr && it < 40) tr[88 + it] = clock64();
            }
            __syncwarp();                                // stay converged: the next blocking wait must be a whole-warp wait
        }
    } else if (warp == 8) {
        // ======================= MMA issuer =====================================
        const uint32_t idesc = make_idesc_bf16(TC_BM, BN);
        // descriptors are linear in the (address >> 4) field: build them once, add offsets per MMA
        const uint64_t dA0 = make_smem_desc_sw128(base + tiles_off);
        const uint64_t dB0 = make_smem_desc_sw128(base + tiles_off + b_off);
#pragma unroll 1
        for (int it = 0; it < n_steps; ++it) {
            const int s = it % stages;
            __syncwarp();                                // converged whole-warp wait (see the producer comment)
            mbar_wait(smem_u32(&ctl->full[s]), (uint32_t)(it / stages) & 1u);
            tc_fence_after();
            if (tr && it == 0 && lane == 0) tr[3] = clock64();
            if (tr && it < 32 && lane == 0) tr[8 + it] = clock64();
            if (lane == 0) {
                const int nu = min(units, n_items - it * units);
#pragma unroll 1
                for (int u = 0; u < nu; ++u) {
                    const uint32_t so = ((uint32_t)s * stage_bytes + (uint32_t)u * unit_bytes) >> 4;
                    const uint64_t da = dA0 + so, db = dB0 + so;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        umma_bf16(tmem, da + 2 * j, db + 2 * j, idesc, (it | u | j) ? 1u : 0u);
                        if (two) umma_bf16(tmem + (uint32_t)BN, da + (a2_off >> 4) + 2 * j, db + (TB >> 4) + 2 * j, idesc, (it | u | j) ? 1u : 0u);
                    }
                }
                umma_commit(smem_u32(&ctl->empty[s]));
            }
            __syncwarp();
        }
        if (lane == 0) { umma_commit(smem_u32(&ctl->accum)); if (tr) tr[4] = clock64(); }
        __syncwarp();
        tc_fence_before();
    } else {
        // ======================= epilogue (warps 0-7) ===========================
        // thread = (tile row t = image, half h).  Its columns, in chunks of 8:
        //   pool: the tile holds ng channels x the 4 pixels of a 2x2 window (column = q*ng + channel); half h owns ng/2
        //         channels = NC chunks, each present once per pixel q
        //   else: the tile's single pixel, columns h*BN/2 + k*8
        constexpr int NCH = BN / 16;                      // 8-column chunks per thread
        const int t = threadIdx.x & 127, h = threadIdx.x >> 7, b = m0 + t;
        const bool bvalid = b < g.B;
        const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        const int nc = p.pool ? NCH / 4 : NCH;            // channel chunks this thread owns
        // chunk index k -> (channel chunk cc, pixel group q): pool: k = cc*4 + q (the four pixels of a chunk are consecutive)
        auto chunk_col = [&](int k, int& q, int& n0) {
            if (p.pool) { const int cc = k >> 2; q = k & 3; n0 = cb * ng + h * (ng >> 1) + cc * 8; return q * ng + h * (ng >> 1) + cc * 8; }
            q = 0; n0 = cb * BN + h * (BN / 2) + k * 8;
            return h * (BN / 2) + k * 8;
        };
        // (1) while the main loop runs: draw this row's LRT noise and park it in tensor memory
        if (philox) {
            int b_s = b;                                 // image index inside its MC sample
            const NoiseKey nkey = fold_key(effective_key(p.key, p.stream_base), p.fold, b, b_s);
#pragma unroll 1
            for (int k = 0; k < NCH; ++k) {
                int q, n0, oh, ow;
                const int c0 = chunk_col(k, q, n0);
                group_pix(q, oh, ow);
                float z8[8];
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (bvalid && n0 + 4 * hh < g.N) z = act_noise4(nkey, b_s, oh * g.OW + ow, n0 + 4 * hh, g.OHW, g.N);
                    z8[4 * hh] = z.x; z8[4 * hh + 1] = z.y; z8[4 * hh + 2] = z.z; z8[4 * hh + 3] = z.w;
                }
                tmem_st8(lane_base + NOISE_COL + (uint32_t)c0, z8);
            }
            tmem_st_wait();
        }
        const bool any_mma = n_items > 0;  // did the schedule of warp 8 contain at least one step?
        // (2) accumulator ready
        pdl_wait();                                      // our output buffers may still be read by the previous step's consumer
        if (threadIdx.x < BN) {                          // bias / bias variance of this tile's columns (written by the prep
            const int c = threadIdx.x;                   // kernel, which may be the programmatic predecessor: after the wait)
            const int n = p.pool ? (cb * ng + (c % ng)) : (cb * BN + c);
            ctl->bias[c] = p.bias_ws[n];
            ctl->bvar[c] = p.bias_ws[p.n_cblk * ng + n];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // the eight epilogue warps only
        mbar_wait(smem_u32(&ctl->accum), 0u);
        tc_fence_after();
        if (tr && threadIdx.x == 0) tr[5] = clock64();
        const int ohw_out = p.pool ? (g.OHW >> 2) : g.OHW;
        (void)nc;
        float r[8];
#pragma unroll 1
        for (int k = 0; k < NCH; ++k) {
            int q, n0;
            const int c0 = chunk_col(k, q, n0);           // tile column / first output channel of this chunk
            float am[8];
            tmem_ld8_nowait(lane_base + (uint32_t)c0, am);
            if (two) {
                float av[8], e8[8];
                tmem_ld8_nowait(lane_base + (uint32_t)BN + (uint32_t)c0, av);
                if (philox) tmem_ld8_nowait(lane_base + NOISE_COL + (uint32_t)c0, e8);
                tmem_ld_wait();
                if (!philox) {
                    int oh, ow;
                    group_pix(q, oh, ow);
#pragma unroll
                    for (int u = 0; u < 8; ++u)
                        e8[u] = (bvalid && n0 + u < g.N) ? __ldg(p.eps_a + ((size_t)b * g.N + n0 + u) * g.OHW + oh * g.OW + ow) : 0.0f;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float var = 1e-16f + ((any_mma ? av[u] : 0.0f) + ctl->bvar[c0 + u]);
                    am[u] = (any_mma ? am[u] : 0.0f) + ctl->bias[c0 + u] + fast_sqrt(var) * e8[u];
                }
            } else {
                tmem_ld_wait();
#pragma unroll
                for (int u = 0; u < 8; ++u) am[u] = (any_mma ? am[u] : 0.0f) + ctl->bias[c0 + u];
            }
            if (p.pool) {                                 // 2x2 max over the chunk's four pixels, store after the last
#pragma unroll
                for (int u = 0; u < 8; ++u) r[u] = q ? fmaxf(r[u], am[u]) : am[u];
                if (q < 3) continue;
            } else {
#pragma unroll
                for (int u = 0; u < 8; ++u) r[u] = am[u];
            }
            if (!bvalid) continue;
#pragma unroll
            for (int u = 0; u < 8; ++u) r[u] = fast_act(r[u], p.act);       // act is monotone: act(max) == max(act)
            if (p.out_mode == OUT_PACKED_BF16) {          // tiled packed (N % 64 == 0 guaranteed by the host)
                const size_t off = tiled_chunk_offset(b, pset * g.N + n0, p.out_pitch >> 6, p.y_sq ? 2 : 1);
                *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.y) + off) =
                    make_uint4(pack_bf16(r[0], r[1]), pack_bf16(r[2], r[3]), pack_bf16(r[4], r[5]), pack_bf16(r[6], r[7]));
                if (p.y_sq)
                    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.y_sq) + off) =
                        make_uint4(pack_bf16(r[0] * r[0], r[1] * r[1]), pack_bf16(r[2] * r[2], r[3] * r[3]),
                                   pack_bf16(r[4] * r[4], r[5] * r[5]), pack_bf16(r[6] * r[6], r[7] * r[7]));
            } else {
                float* yo = reinterpret_cast<float*>(p.y);
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int n = n0 + u;
                    if (n < g.N) {
                        if (p.out_mode == OUT_ROWMAJOR_F32) yo[((size_t)b * ohw_out + pset) * g.N + n] = r[u];
                        else yo[((size_t)b * g.N + n) * ohw_out + pset] = r[u];
                    }
                }
            }
        }
        if (tr && threadIdx.x == 0) tr[6] = clock64();
        tc_fence_before();
    }
    __syncthreads();
    tc_fence_after();
    if (warp == 8) tmem_dealloc(tmem, tmem_cols);
    if (tr && threadIdx.x == 256) tr[7] = clock64();
    tl_exit(p.tl_gemm, 256);
}

// ------------------------------------------------------------- host side
inline bool fused_supported(const Geom& g, int pool) {
    if (g.DH != 1 || g.DW != 1) return false;
    if (g.HW > 64) return false;                       // "small map" regime
    if (pool && ((g.OH & 1) || (g.OW & 1))) return false;
    if (g.Cin % 64) return false;                      // tiled packed input: whole 64-column blocks per pixel
    if ((long)g.HW * (g.Cin / 64) > TAP_MAX_ITEMS) return false;
    return true;
}

inline size_t prep2_smem_bytes(int planes, int khw, int r) { return (size_t)planes * khw * prep2_slab(r) * 2; }

// The launch configuration of one tap-GEMM step: launch_fused runs exactly this, and bbb_debug_fused_config reports it.
struct TapConfig {
    int bn;            // tile width: 64 or 128 output columns
    int ng;            // output channels per column group (bn, or bn / 4 with the pool: four pixels per tile)
    int n_cblk, n_kblk;
    int two_per_sm;    // BN = 64 with more CTAs than SMs: tap_gemm_kernel<2, 64>, two resident CTAs per SM
    int prep_conv;     // the prep is tap_prep_conv_kernel (else tap_prep_kernel)
    int prep_rows;     // tap_prep_conv_kernel: output channels per CTA
};

inline TapConfig tap_config(const Geom& g, int planes, int pool, int prev_hw, int n_sm, bool prefer_wide) {
    TapConfig c;
    // tile width: 128 columns when Cout allows it and the grid still covers most of the machine (operand bytes per MAC,
    // see tap_gemm_kernel) -- or always when the caller keeps several steps in flight (bbb_set_wide_tiles) -- else 64.  BBB_B200_TAP_BN=64 forces the narrow tile (A/B measurements).
    const int psets = pool ? (g.OH / 2) * (g.OW / 2) : g.OHW;
    const int row_tiles = (g.B + TC_BM - 1) / TC_BM;
    c.bn = 64;
    {
        static const int force = [] { const char* e = getenv("BBB_B200_TAP_BN"); return e ? atoi(e) : 0; }();
        const int ng128 = pool ? 32 : 128;
        if (g.N % ng128 == 0 && (prefer_wide || (long)psets * (g.N / ng128) * row_tiles >= (long)n_sm * 6 / 10)) c.bn = 128;
        if (force == 64 || force == 128) c.bn = (force == 128 && g.N % ng128 == 0) ? 128 : 64;
    }
    c.ng = pool ? c.bn / 4 : c.bn;
    c.n_cblk = (g.N + c.ng - 1) / c.ng;
    c.n_kblk = (g.Cin + 63) / 64;
    // conv layers: the coalesced prep variant (rows x 64-channel block per CTA); R = rows per CTA, shrunk until the
    // grid covers the SMs and the staging tile fits 48 KB
    static const bool prep2_on = [] { const char* e = getenv("BBB_B200_PREP2"); return !(e && e[0] == '0'); }();
    int R = 8;
    const int npad = c.n_cblk * c.ng;
    // <= 26 KB of staging per CTA: the preps run beside the GEMM chain (side streams) and must fit next to its CTAs
    constexpr size_t kPrepSmem = 26 * 1024;
    // (smaller CTAs -- >= 4 per SM -- were tried for more loads in flight: the preps then lose the scheduling race against
    //  the high-priority GEMM chain and the third layer's prep finished at 61 us instead of 21 us: 123 vs 107 us per step)
    while (R > 2 && ((long)(npad / R) * c.n_kblk < n_sm || prep2_smem_bytes(planes, g.KHW, R) > kPrepSmem)) R >>= 1;
    c.prep_rows = R;
    c.prep_conv = prep2_on && g.KHW > 1 && prev_hw == 1 && g.Cin % 64 == 0 && prep2_smem_bytes(planes, g.KHW, R) <= 48 * 1024;
    // Configurations.  BN = 64: (A) one CTA per SM, stage = 2 K blocks, deep ring; (B) two CTAs per SM (~99 KB each) when
    // the grid has more CTAs than SMs, so that all tiles run in ONE wave and one CTA's epilogue overlaps the other's main
    // loop.  BN = 128: one CTA per SM, 64 KB (LRT) / 32 KB K blocks, three stages.
    const long n_ctas = (long)psets * c.n_cblk * row_tiles;
    c.two_per_sm = c.bn == 64 && n_ctas > n_sm;
    return c;
}

inline cudaError_t launch_fused(FusedArgs a, const void* x, const void* x_sq, cudaStream_t st, int* n_launch, const char** why,
                                bool do_prep = true, bool do_gemm = true, int n_sm = 148, bool prefer_wide = false) {
    const Geom& g = a.g;
    *n_launch = 0;
    a.planes = tc_planes(a.variant, a.sample);
    const TapConfig cfg = tap_config(g, a.planes, a.pool, a.prev_hw, n_sm, prefer_wide);
    const int psets = a.pool ? (g.OH / 2) * (g.OW / 2) : g.OHW;
    const int row_tiles = (g.B + TC_BM - 1) / TC_BM;
    const int bn = cfg.bn;
    a.ng = cfg.ng;
    a.n_cblk = cfg.n_cblk;
    a.n_kblk = cfg.n_kblk;
    a.taps = g.KHW;
    const bool lrt = a.variant == BBB_VARIANT_LRT;
    a.x = x; a.x_sq = x_sq;
    if (do_gemm && a.planes == 2 && x_sq != (const void*)((const __nv_bfloat16*)x + 128 * 64)) {
        *why = "LRT fused layer needs the activation with interleaved x / x^2 blocks (x_sq == x + 8192 elements)";
        return cudaErrorInvalidValue;
    }
    if (do_prep) {
        const long items = (long)a.taps * a.n_cblk * a.n_kblk * a.ng * 8;
        int grid = (int)((items + 255) / 256);
        if (grid > 2048) grid = 2048;
        if (grid < 1) grid = 1;
        static const bool carve = [] {           // see launch_fwd_tc: keep every kernel of the chain on one smem carve-out
            const char* e = getenv("BBB_B200_PREP_CARVEOUT");
            if (e && e[0] == '0') return false;
            cudaFuncSetAttribute(tap_prep_kernel<BBB_VARIANT_LRT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            cudaFuncSetAttribute(tap_prep_kernel<BBB_VARIANT_BBB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            return true;
        }();
        (void)carve;
        const int R = cfg.prep_rows, npad = a.n_cblk * a.ng;
        const size_t need = prep2_smem_bytes(a.planes, g.KHW, R);
        if (cfg.prep_conv) {
            static const bool carve2 = [] {
                const char* e = getenv("BBB_B200_PREP_CARVEOUT");
                if (e && e[0] == '0') return false;
                cudaFuncSetAttribute(tap_prep_conv_kernel<BBB_VARIANT_LRT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
                cudaFuncSetAttribute(tap_prep_conv_kernel<BBB_VARIANT_BBB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
                return true;
            }();
            (void)carve2;
            int grid2 = (npad / R) * a.n_kblk;
            if (grid2 > 2048) grid2 = 2048;
            if (lrt) tap_prep_conv_kernel<BBB_VARIANT_LRT><<<grid2, 256, need, st>>>(a, R);
            else     tap_prep_conv_kernel<BBB_VARIANT_BBB><<<grid2, 256, need, st>>>(a, R);
        }
        else if (lrt) tap_prep_kernel<BBB_VARIANT_LRT><<<grid, 256, 0, st>>>(a);
        else          tap_prep_kernel<BBB_VARIANT_BBB><<<grid, 256, 0, st>>>(a);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        *n_launch += 1;
    }
    if (!do_gemm) return cudaSuccess;
    // (configurations: see tap_config.)  The LRT noise tile always lives in tensor memory and is drawn during the main loop.
    const bool two_per_sm = cfg.two_per_sm != 0;
    int stages;
    if (bn == 128)       { stages = 3; a.units = a.planes == 2 ? 1 : 2; }
    else if (two_per_sm) { stages = 2; a.units = a.planes == 2 ? 1 : 2; }
    else                 { stages = a.planes == 2 ? 2 : 4; a.units = TAP_UNITS; }
    if (const char* e = getenv("BBB_B200_STAGES")) { const int v = atoi(e); if (v >= 2 && v <= stages) stages = v; }
    const size_t unit_bytes = (size_t)a.planes * (TC_A_BYTES + (size_t)bn * 128);
    const size_t smem = 1023 + 2048 + (size_t)stages * a.units * unit_bytes;   // align slack + control/schedule + ring
    dim3 grid(psets * a.n_cblk, row_tiles);
    cudaError_t e;
    auto launch = [&](auto kernel) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaError_t e2 = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e2 != cudaSuccess) return e2;
        return launch_pdl(kernel, grid, dim3(TAP_THREADS), smem, st, a, stages);
    };
    e = bn == 128 ? launch(tap_gemm_kernel<1, 128>) : (two_per_sm ? launch(tap_gemm_kernel<2, 64>) : launch(tap_gemm_kernel<1, 64>));
    if (e != cudaSuccess) return e;
    e = cudaGetLastError();
    if (e == cudaSuccess) *n_launch += 1;
    return e;
}

}  // namespace bbb
