// K3: full-catalog scoring fused with mask + top-k as a CERTIFIED FILTER on the tensor cores.
//
// The score matrix (115 MB per 4096 users at 7k items, 16 GB at 1M) is never written and no threshold depends on
// timing.  The tensor cores (tcgen05, kind::f16, ONE pass over operands rounded to fp16 after a power-of-two scaling:
// the same 11-bit significand as tf32 at twice the MMA rate and half the operand bytes) compute APPROXIMATE scores
// s~ with a proven bound |s~ - s| <= eps * |u| * max|i| (+ a subnormal term that only matters for degenerate
// tables, see cf_thr_kernel); they are only used to decide which (user, item) pairs can
// be in the top-k.  Every pair that can is then scored again in full fp32 (fmaf chain, the arithmetic of the exact
// kernel below), and the final order is taken on those fp32 values -- so the result is the fp32 top-k, tie -> lower
// item index, exactly the contract of topk.cu.
//
//   cf_pack_kernel      operands -> fp16 (round to nearest) in the UMMA canonical K-major no-swizzle layout, tiles of
//                       128 rows, scaled by a power of two (per user row; one for the whole catalogue) so that the
//                       largest element lands in [2^14, 2^15): no overflow, and fp16 subnormals only for elements
//                       2^-28 below the largest.  Scores, norms and thresholds of a row all live in that scaled domain
//                       (the exact re-scoring reads the original tables).  Row norms (users) / maximum row norm
//                       (catalogue).  The catalogue side is packed once per embedding table (mmrec_catalog_pack_f32).
//   cf_pass_kernel<1>   s~ for every (user, item); epilogue = maximum of every group of w = 16 gw consecutive items
//                       (tcgen05.ld -> FMNMX3 tree), written as gmax[row][group].  No branches, no atomics.
//   cf_thr_kernel       per row: t = the need-th largest group maximum, need = k + (masked items of the row).  At
//                       least `need` distinct items have s~ >= t, so >= k unmasked ones have s >= t - eps'; hence every
//                       member of the true top-k has s~ >= thr = t - 2 eps'.
//   cf_pass_kernel<2>   s~ again (same instructions, same bits); epilogue = one bit per score, s~ >= thr, 128 bits per
//                       (row, item tile) written as one 16-byte store.  ~ (need + a few) bits per row are set.
//   cf_final_kernel     per row (one warp): the set bits -> drop masked items -> exact fp32 score from the ORIGINAL
//                       tables -> rank on (value desc, item asc) -> top-k.
//   cf_exact_kernel     rows the filter cannot serve (need > number of groups, > CF_CAP candidates, non-finite scores):
//                       all items in fp32 on CUDA cores + radix select; exits at once when no row is flagged.
// Work distribution of the passes: a unit = (pair of 128-user tiles, 128-item tile); the units are dealt to the CTAs
// (one per SM) in contiguous runs, so every SM gets the same number of units whatever the batch size (no wave
// quantisation), a 256-user operand stays resident while its run of item tiles streams through a bulk-copy ring, and
// every item slab read from L2 feeds two MMAs (32 B/cycle/SM at full tensor rate; one 128-user tile per CTA would
// need 64, more than L2 delivers to 148 SMs).
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cub/device/device_scan.cuh>

#include "tc_common.cuh"

namespace mmrec {

using namespace tc;

constexpr int CF_TILE = 128;                    // rows of one MMA operand tile (users: TMEM lanes; items: TMEM columns)
// An item slab is the whole K of a 128-item tile (8 / 16 / 32 KB at KP = 32 / 64 / 128): one barrier round trip per unit.
constexpr int CF_EPI_WARPS = 16;                // (buffer parity, user half, TMEM lane quarter)
constexpr int CF_THREADS = 64 + 32 * CF_EPI_WARPS;
constexpr int CF_MAX_STAGES = 10;
constexpr int CF_CAP = 512;                     // candidates one warp ranks per row
constexpr int CF_EX_SLOTS = 128;                // CTAs (and key buffers) of the exact kernel
constexpr float CF_EPS = 1.125f / 1024.f;       // |s~ - s| <= CF_EPS |u| |i|: two RN roundings to 11 significand bits (2^-11 each) + accumulation slack
constexpr float CF_EPS_SUB = 1.0f / 16777216.f; // fp16 subnormal spacing 2^-24 (scaled domain): |dx| <= 2^-11 |x| + 2^-25 per element

struct CfSmem {
    uint32_t a, slab0, slab, bars, tmem_ptr, total;
    int stages;
};
__host__ __device__ inline CfSmem cf_smem(int KP) {
    CfSmem L;
    L.a = 0;
    L.slab0 = 2 * CF_TILE * KP * 2;             // the 256-user operand: two tiles of 128 rows, fp16
    const uint32_t slab = CF_TILE * KP * 2;
    L.slab = slab;
    L.stages = (int)((226u * 1024u - L.slab0 - 300u) / slab);        // as many slabs in flight as shared memory holds
    if (L.stages > CF_MAX_STAGES) L.stages = CF_MAX_STAGES;
    L.bars = L.slab0 + L.stages * slab;
    L.tmem_ptr = L.bars + 32 * 8;
    L.total = L.tmem_ptr + 16;
    return L;
}
// barrier slots
enum { CB_AFULL = 0, CB_AFREE = 1, CB_FULL = 2, CB_EMPTY = 2 + CF_MAX_STAGES, CB_TFULL = 2 + 2 * CF_MAX_STAGES, CB_TEMPTY = 4 + 2 * CF_MAX_STAGES };

struct CfParams {
    const char* Upk;                            // fp16 [pairs][2][KP/8][16][8][8]
    const char* Ipk;                            // fp16 [item tiles][KP/8][16][8][8]
    int KP, n_it;
    int64_t B, n_items, n_units;
    float* gmax; int G, gw;                     // pass 1: [B][G], G = n_it * (8 / gw)
    const float* thr; uint4* bitmap;            // pass 2: [B], [B][n_it]
    int dbg;                                    // tuning aid (env MMREC_CF_DEBUG): 1 = epilogue skips its TMEM loads, 2 = no MMAs issued
};

__device__ __forceinline__ void cf_tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
// wait for the outstanding tcgen05.ld of this thread; the registers are operands so that no use of them can be
// scheduled above the wait
__device__ __forceinline__ void cf_tmem_wait16(uint32_t (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :: "memory");
}
__device__ __forceinline__ void cf_tmem_ld32(uint32_t taddr, uint32_t (&a)[16], uint32_t (&b)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]),
          "=r"(a[8]), "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]),
          "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]), "=r"(b[4]), "=r"(b[5]), "=r"(b[6]), "=r"(b[7]),
          "=r"(b[8]), "=r"(b[9]), "=r"(b[10]), "=r"(b[11]), "=r"(b[12]), "=r"(b[13]), "=r"(b[14]), "=r"(b[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void cf_tmem_wait32(uint32_t (&a)[16], uint32_t (&b)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                   "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                   "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                   "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15])
                 :: "memory");
}
__device__ __forceinline__ float cf_max3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
__device__ __forceinline__ float cf_max16(const uint32_t (&v)[16]) {
#define CF_F(i) __uint_as_float(v[i])
    const float a = cf_max3(CF_F(0), CF_F(1), CF_F(2)), b = cf_max3(CF_F(3), CF_F(4), CF_F(5)), c = cf_max3(CF_F(6), CF_F(7), CF_F(8));
    const float d = cf_max3(CF_F(9), CF_F(10), CF_F(11)), e = cf_max3(CF_F(12), CF_F(13), CF_F(14));
    return fmaxf(cf_max3(a, b, c), cf_max3(d, e, CF_F(15)));
#undef CF_F
}
// 16 scores -> 16 bits, bit (15 - j) = (v[j] < thr): sign of the (exact, Sterbenz) difference, shifted in by a funnel
// shift -- FADD on the fma pipe, SHF on the alu pipe, two chains for ILP
__device__ __forceinline__ uint32_t cf_lt16(const uint32_t (&v)[16], float thr) {
    uint32_t a = 0, b = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        a = __funnelshift_l(__float_as_uint(__uint_as_float(v[j]) - thr), a, 1);
        b = __funnelshift_l(__float_as_uint(__uint_as_float(v[8 + j]) - thr), b, 1);
    }
    return ((a & 0xffu) << 8) | (b & 0xffu);
}

// ---- producer: the 256-user operand of the current pair, then its run of item slabs ----------------------------
__device__ __forceinline__ void cf_producer(const CfParams& p, const CfSmem& L, uint32_t sbase, int64_t u0, int64_t u1) {
    const uint32_t bar = sbase + L.bars;
    const uint32_t a_bytes = 2 * CF_TILE * p.KP * 2;
    const uint32_t piece = L.slab < 16384u ? L.slab : 16384u;        // bulk copies of at most 16 KB
    // (pair, it) and the ring position advance by counting: a 64-bit division per unit is several hundred cycles of a
    // single thread's dependent instructions, and this loop is what the slab ring's refill rate hangs on
    int64_t pair = u0 / p.n_it;
    int it = (int)(u0 - pair * p.n_it);
    bool new_pair = true;
    uint32_t a_cnt = 0, slot = 0, ph = 1;                            // ph: parity to wait for on the slot's "empty" barrier
    for (int64_t u = u0; u < u1; ++u) {
        if (new_pair) {
            if (a_cnt > 0) mbar_wait(bar + CB_AFREE * 8, (a_cnt - 1) & 1);   // every MMA that reads the old operand is done
            mbar_expect_tx(bar + CB_AFULL * 8, a_bytes);
            const char* src = p.Upk + pair * (int64_t)a_bytes;
            for (uint32_t o = 0; o < a_bytes; o += 16384) bulk_g2s(sbase + L.a + o, src + o, 16384, bar + CB_AFULL * 8);
            ++a_cnt;
            new_pair = false;
        }
        const char* src = p.Ipk + (int64_t)it * L.slab;
        const uint32_t fb = bar + (CB_FULL + slot) * 8;
        mbar_wait(bar + (CB_EMPTY + slot) * 8, ph);
        if (p.dbg & 16) {                                             // (tuning aid: no item traffic)
            mbar_arrive(fb);
        } else {
            mbar_expect_tx(fb, L.slab);
            const uint32_t dst = sbase + L.slab0 + slot * L.slab;
            for (uint32_t o = 0; o < L.slab; o += piece) bulk_g2s(dst + o, src + o, piece, fb);
        }
        if (++slot == (uint32_t)L.stages) { slot = 0; ph ^= 1; }
        if (++it == p.n_it) { it = 0; ++pair; new_pair = true; }
    }
}

// ---- MMA issuer: one thread, M128 N128 K16 (kind::f16), two user halves per item slab ------------------------------
__device__ __forceinline__ void cf_mma(const CfParams& p, const CfSmem& L, uint32_t sbase, uint32_t tmem_base, int64_t u0, int64_t u1) {
    const uint32_t bar = sbase + L.bars;
    constexpr uint32_t LBO = (CF_TILE / 8) * 128, SBO = 128;         // both operands: tiles of 128 rows
    const uint32_t idesc = idesc_f16(CF_TILE, CF_TILE);
    const int ksteps = p.KP / 16;
    const uint32_t half_bytes = CF_TILE * p.KP * 2;
    uint32_t a_cnt = 0;
    int halves = 2;
    // The issuing thread is a single instruction stream: measured (tools/probe_mma.py) ~200 cycles per tcgen05.mma when
    // the descriptors are rebuilt around every instruction -- twice what the tensor pipe needs for M128 N128.  So the
    // descriptors are built once and only their address field (low word, 16-byte units) moves.
    const uint64_t a_desc0 = smem_desc(sbase + L.a, LBO, SBO), a_desc1 = smem_desc(sbase + L.a + half_bytes, LBO, SBO);
    const uint64_t b_desc0 = smem_desc(sbase + L.slab0, LBO, SBO);
    const uint64_t kstep = (2 * LBO) >> 4;                           // one K step of 16 = two 16-byte k blocks
    int64_t pair = u0 / p.n_it;
    int it = (int)(u0 - pair * p.n_it);
    bool new_pair = true;
    uint32_t slot = 0, ph = 0, buf = 0, tph = 1;                      // ring position / parity; accumulator buffer / its "empty" parity
    uint64_t bd_slot = b_desc0;
    const uint64_t slab_step = L.slab >> 4;
    for (int64_t u = u0; u < u1; ++u) {
        mbar_wait(bar + (CB_TEMPTY + buf) * 8, tph);                  // accumulators drained by the epilogue
        if (new_pair) {
            mbar_wait(bar + CB_AFULL * 8, a_cnt & 1);
            ++a_cnt;
            halves = (pair * 2 * CF_TILE + CF_TILE < p.B) ? 2 : 1;
            new_pair = false;
        }
        mbar_wait(bar + (CB_FULL + slot) * 8, ph);
        if (!(p.dbg & 64)) fence_after_sync();
        const uint32_t d0 = tmem_base + (buf * 2 + 0) * CF_TILE, d1 = d0 + CF_TILE;
        uint64_t ad0 = a_desc0, ad1 = a_desc1, bd = bd_slot;
        if (!(p.dbg & 2)) {
            if (halves == 2) {
#pragma unroll 4
                for (int j = 0; j < ksteps; ++j) {
                    mma_f16(d0, ad0, bd, idesc, j ? 1u : 0u);
                    mma_f16(d1, ad1, bd, idesc, j ? 1u : 0u);
                    ad0 += kstep; ad1 += kstep; bd += kstep;
                }
            } else {
#pragma unroll 4
                for (int j = 0; j < ksteps; ++j) {
                    mma_f16(d0, ad0, bd, idesc, j ? 1u : 0u);
                    ad0 += kstep; bd += kstep;
                }
            }
        }
        if (p.dbg & 32) {                                             // (tuning aid, only meaningful without MMAs: plain arrives)
            mbar_arrive(bar + (CB_EMPTY + slot) * 8);
            mbar_arrive(bar + (CB_TFULL + buf) * 8);
        } else {
            mma_commit(bar + (CB_EMPTY + slot) * 8);                  // slab consumed -> slot back to the producer
            mma_commit(bar + (CB_TFULL + buf) * 8);                   // accumulators complete -> epilogue
        }
        bd_slot += slab_step;
        if (++slot == (uint32_t)L.stages) { slot = 0; ph ^= 1; bd_slot = b_desc0; }
        if (++it == p.n_it) { it = 0; ++pair; new_pair = true; }
        if (new_pair || u + 1 == u1) mma_commit(bar + CB_AFREE * 8);
        buf ^= 1;
        if (buf == 0) tph ^= 1;
    }
}

// ---- epilogue: thread = one user row, 128 accumulator columns per unit in 8 chunks of 16, loads one chunk ahead --------
template <int PASS, int GPT>
__device__ __forceinline__ void cf_epilogue(const CfParams& p, const CfSmem& L, uint32_t sbase, uint32_t tmem_base, int u0, int u1,
                                            int e, int lane) {
    const uint32_t bar = sbase + L.bars;
    const int q = (e + 2) & 3;                                       // = warp % 4: the TMEM lane quarter this warp may read
    const int h = (e >> 2) & 1, par = e >> 3;
    constexpr int gpt = GPT;                                          // groups per item tile (pass 1): 8 / gw
    int cur_pair = -1;
    int64_t row = 0;
    bool live = false;
    float thr = INFINITY;
    int pair = (u0 + par) / p.n_it;
    int it = (u0 + par) - pair * p.n_it;
    uint32_t fph = 0;
    for (int u = u0 + par; u < u1; u += 2, fph ^= 1) {
        if (pair != cur_pair) {
            cur_pair = pair;
            row = (int64_t)pair * (2 * CF_TILE) + h * CF_TILE + q * 32 + lane;
            live = row < p.B;
            if (PASS == 2) thr = live ? __ldg(p.thr + row) : INFINITY;
        }
        mbar_wait(bar + (CB_TFULL + par) * 8, fph);
        fence_after_sync();
        // (a whole half beyond the batch: nothing to read, but the buffer still has to be released)
        if ((int64_t)pair * (2 * CF_TILE) + h * CF_TILE < p.B && !(p.dbg & 1)) {
            const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + (par * 2 + h) * CF_TILE;
            const int n_valid = (int)(p.n_items - (int64_t)it * CF_TILE);      // < 128 on the last tile only
            uint32_t va[16], vb[16];
            float gm[8];
            uint32_t w[4];
#pragma unroll
            for (int c = 0; c < 8; c += 2) {
                // 32 columns per tcgen05.ld (MMREC_CF_DEBUG bit 2: 16 per load, the next one requested before this one is used)
                if (p.dbg & 4) {
                    if (c == 0) cf_tmem_ld16(t0, va);
                    cf_tmem_wait16(va);
                    cf_tmem_ld16(t0 + (c + 1) * 16, vb);
                } else {
                    cf_tmem_ld32(t0 + c * 16, va, vb);
                    cf_tmem_wait32(va, vb);
                }
                if (n_valid < CF_TILE) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (c * 16 + j >= n_valid) va[j] = 0xff800000u;          // -inf: never a maximum, never a hit
                }
                if (PASS == 1) gm[c] = cf_max16(va);
                const uint32_t lt0 = PASS == 2 ? cf_lt16(va, thr) : 0u;
                if (p.dbg & 4) {
                    cf_tmem_wait16(vb);
                    if (c + 2 < 8) cf_tmem_ld16(t0 + (c + 2) * 16, va);
                }
                if (n_valid < CF_TILE) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if ((c + 1) * 16 + j >= n_valid) vb[j] = 0xff800000u;
                }
                if (PASS == 1) {
                    gm[c + 1] = cf_max16(vb);
                    if (gpt <= 4) gm[c] = fmaxf(gm[c], gm[c + 1]);    // groups of 32 items and wider: fold as we go
                    if (gpt == 8 && (c & 2) && live)                  // groups of 16: four maxima are a 16-byte store
                        reinterpret_cast<float4*>(p.gmax + row * p.G + (int64_t)it * 8)[c >> 2] = make_float4(gm[c - 2], gm[c - 1], gm[c], gm[c + 1]);
                }
                if (PASS == 2) w[c >> 1] = ~((lt0 << 16) | cf_lt16(vb, thr));   // bit (31 - j) of word (c / 2): column 32 (c / 2) + j passes
            }
            if (live) {
                if (PASS == 1) {
                    float* dst = p.gmax + row * p.G + (int64_t)it * gpt;
                    if (gpt == 8) {
                        // (stored inside the loop)
                    } else if (gpt == 4) {
                        *reinterpret_cast<float4*>(dst) = make_float4(gm[0], gm[2], gm[4], gm[6]);
                    } else if (gpt == 2) {
                        *reinterpret_cast<float2*>(dst) = make_float2(fmaxf(gm[0], gm[2]), fmaxf(gm[4], gm[6]));
                    } else {
                        *dst = fmaxf(fmaxf(gm[0], gm[2]), fmaxf(gm[4], gm[6]));
                    }
                } else {
                    p.bitmap[row * p.n_it + it] = make_uint4(w[0], w[1], w[2], w[3]);
                }
            }
        }
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar + (CB_TEMPTY + par) * 8);
        it += 2;
        while (it >= p.n_it) { it -= p.n_it; ++pair; }
    }
}

template <int PASS, int GPT>
__global__ void __launch_bounds__(CF_THREADS, 1) cf_pass_kernel(const CfParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const CfSmem L = cf_smem(p.KP);
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar = sbase + L.bars;
    if (threadIdx.x == 0) {
        for (int i = 0; i < CB_TEMPTY; ++i) mbar_init(bar + i * 8, 1);
        mbar_init(bar + CB_TEMPTY * 8, 8); mbar_init(bar + (CB_TEMPTY + 1) * 8, 8);   // 2 halves x 4 lane quarters release a buffer pair
        mbar_fence_init();
    }
    if (warp == 1) { tmem_alloc(sbase + L.tmem_ptr, 512); tmem_relinquish(); }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + L.tmem_ptr);
    // contiguous run of units for this CTA
    const int64_t u0 = (int64_t)blockIdx.x * p.n_units / gridDim.x;
    const int64_t u1 = (int64_t)(blockIdx.x + 1) * p.n_units / gridDim.x;
    if (warp == 0) {
        if (lane == 0) cf_producer(p, L, sbase, u0, u1);
    } else if (warp == 1) {
        if (lane == 0) cf_mma(p, L, sbase, tmem_base, u0, u1);
    } else {
        cf_epilogue<PASS, GPT>(p, L, sbase, tmem_base, (int)u0, (int)u1, warp - 2, lane);
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------------------------
// operand packing
// ------------------------------------------------------------------------------------------------------------------
// Power of two that brings a largest magnitude m into [2^14, 2^15) (m = 0, inf, NaN, or below 2^-113: 1 -- the
// non-finite cases flag their rows in cf_thr_kernel; the tiny ones are what CF_EPS_SUB in the margin is for).
__device__ __forceinline__ float cf_scale_for(uint32_t m_bits) {
    const uint32_t e = (m_bits >> 23) & 0xffu;                       // biased exponent
    if (e == 0u || e == 255u || e < 14u) return 1.0f;
    return __uint_as_float((268u - e) << 23);                        // 2^(14 - (e - 127))
}

// One thread per (padded row, k block of 8): scale, round to fp16, store 16 bytes into the tile layout; the KP/8 threads
// of a row are consecutive lanes and reduce, with shuffles, the row's largest magnitude (user rows) and then the squared
// norm of the SCALED row.  `scale_src` = the catalogue-wide largest magnitude (items), or NULL: per-row scale (users).
// The norm is taken after scaling so that it is valid for every finite row: the largest scaled element lies in
// [2^14, 2^15), so a user row's sum of squares lies in [2^28, 2^37) whatever the magnitude of its elements (squares of the
// unscaled elements underflow to 0 below ~1e-23 and overflow above ~2e18 at d = 64).  A catalogue row far below the
// catalogue's largest element may underflow here, but such a row does not set the maximum norm.
__device__ __forceinline__ void cf_pack_one(int64_t t, int64_t n_rows, const int64_t* __restrict__ idx, const float* __restrict__ E, int64_t ld,
                                            int d, int KP, const uint32_t* __restrict__ scale_src, uint4* __restrict__ out,
                                            float* __restrict__ row_norm, uint32_t* __restrict__ max_norm) {
    const int kblks = KP / 8;
    const int64_t row = t / kblks;
    const int kb = (int)(t % kblks);
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = 0.f;
    if (row < n_rows) {
        const float* src = E + (idx ? idx[row] : row) * ld;
#pragma unroll
        for (int e = 0; e < 8; ++e)
            if (kb * 8 + e < d) x[e] = __ldg(src + kb * 8 + e);
    }
    uint32_t am;
    if (scale_src) {
        am = __ldg(scale_src);
    } else {
        am = 0u;                                                      // largest |x| as a bit pattern (orders like the value; NaN above inf)
#pragma unroll
        for (int e = 0; e < 8; ++e) { const uint32_t b = __float_as_uint(x[e]) & 0x7fffffffu; am = b > am ? b : am; }
        for (int o = kblks / 2; o > 0; o >>= 1) {
            const uint32_t a2 = __shfl_xor_sync(0xffffffffu, am, o);
            am = a2 > am ? a2 : am;
        }
    }
    const float sc = cf_scale_for(am);
    float ss = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) { x[e] *= sc; ss = fmaf(x[e], x[e], ss); }
    for (int o = kblks / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const __half2 h = __floats2half2_rn(x[2 * e], x[2 * e + 1]);
        w[e] = *reinterpret_cast<const uint32_t*>(&h);
    }
    const int64_t tile = row / CF_TILE;
    const int rr = (int)(row % CF_TILE);
    out[((tile * kblks + kb) * (CF_TILE / 8) + rr / 8) * 8 + (rr % 8)] = make_uint4(w[0], w[1], w[2], w[3]);
    if (kb == 0 && row < n_rows) {
        // Rounded up so that the bound holds: ss sums at most 128 non-negative terms, and each term goes through at most
        // 12 roundings (8 in the thread's fmaf chain, 4 in the shuffle tree at KP = 128), so ss is within 12 2^-24 = 7.2e-7
        // of the exact sum; its square root is within 3.6e-7, plus 2^-24 for sqrtf and 2^-24 for the product: < 1e-6.
        const float nrm = sqrtf(ss) * (1.0f + 1e-6f);
        if (row_norm) row_norm[row] = nrm;
        if (max_norm) atomicMax(max_norm, __float_as_uint(nrm));      // non-negative floats order like their bit patterns
    }
}

// header: word 0 = running maximum (scaled) norm, word 4 = largest magnitude of the table, both zeroed by a memset node
// before the launches; thread 0 of the pack kernel fills in the rest
__global__ void __launch_bounds__(256) cf_item_absmax_kernel(int64_t n_items, const float* __restrict__ Ie, int64_t ldi, int d,
                                                             uint32_t* __restrict__ header) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * 8;
    uint32_t m = 0;
    for (int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); r < n_items; r += warps)        // warp per row
        for (int c = lane; c < d; c += 32) {
            const uint32_t b = __float_as_uint(__ldg(Ie + r * ldi + c)) & 0x7fffffffu;             // |x|; NaN patterns sort above inf
            m = b > m ? b : m;
        }
    m = __reduce_max_sync(0xffffffffu, m);
    if (lane == 0 && m) atomicMax(header + 4, m);
}

__global__ void __launch_bounds__(256) cf_pack_items_kernel(int64_t n_items, const float* __restrict__ Ie, int64_t ldi, int d, int KP,
                                                            uint4* __restrict__ Ipk, uint32_t* __restrict__ header, int64_t n_threads) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_threads) return;                                       // (n_threads is a multiple of 32: whole warps leave together)
    if (t == 0) { header[1] = (uint32_t)n_items; header[2] = (uint32_t)d; header[3] = (uint32_t)KP; }
    cf_pack_one(t, n_items, nullptr, Ie, ldi, d, KP, header + 4, Ipk, nullptr, header);
}

// ---- mask CSR over batch rows -------------------------------------------------------------------------------------
// The reference's evaluation loader emits the mask row-major (batch row ascending: src/utils/dataloader.py:370-391 builds
// it user by user), so the common case is a sorted row array: the row pointers are the positions where the row
// changes, checked as we go, one fully parallel pass.  If any block saw a descent, mask_csr_small_kernel (one CTA:
// count in shared memory, scan, fill) redoes the job for arbitrary order; otherwise it exits at once.
__device__ __forceinline__ void cf_mask_sorted_block(int64_t blk, int64_t nnz, const int64_t* __restrict__ rows, const int64_t* __restrict__ cols,
                                                     int B, int64_t item_offset, int32_t* __restrict__ ptr, int32_t* __restrict__ items,
                                                     int32_t* __restrict__ unsorted) {
    const int64_t j = blk * (int64_t)blockDim.x + threadIdx.x;        // entry j, plus one sentinel thread j == nnz
    int bad = 0;
    if (j <= nnz) {
        const int64_t rj = j < nnz ? rows[j] : (int64_t)B;
        const int64_t rp = j > 0 ? rows[j - 1] : -1;
        bad = j < nnz && rp > rj;
        if (j < nnz) items[j] = (int32_t)(cols[j] - item_offset);
        // rows (rp, rj] start at entry j (rows outside [0, B) own no pointer; clamped so that they delimit correctly)
        const int64_t lo = rp < -1 ? -1 : (rp > B ? B : rp), hi = rj < -1 ? -1 : (rj > B ? B : rj);
        for (int64_t r = lo + 1; r <= hi; ++r) ptr[r] = (int32_t)j;
    }
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) unsorted[blk] = bad;
}

constexpr int MC_MAX_ROWS = 8192;
constexpr int MC_THREADS = 1024;
__global__ void __launch_bounds__(MC_THREADS) mask_csr_small_kernel(int64_t nnz, const int64_t* __restrict__ rows,
                                                                    const int64_t* __restrict__ cols, int B, int64_t item_offset,
                                                                    int32_t* __restrict__ ptr, int32_t* __restrict__ items,
                                                                    const int32_t* __restrict__ unsorted, int n_unsorted) {
    extern __shared__ int32_t mc_sm[];                               // count / cursor [B + 1] | warp totals [32]
    {   // runs only when the sorted pass found the rows out of order (it then left garbage behind)
        int any = 0;
        for (int i = threadIdx.x; i < n_unsorted; i += MC_THREADS) any |= unsorted[i];
        if (!__syncthreads_or(any)) return;
    }
    int32_t* cnt = mc_sm;
    int32_t* wtot = mc_sm + B + 1;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (int r = tid; r <= B; r += MC_THREADS) cnt[r] = 0;
    __syncthreads();
    constexpr int MC_U = 8;                                          // loads in flight per thread (the loop is latency-bound)
    for (int64_t jb = 0; jb < nnz; jb += (int64_t)MC_U * MC_THREADS) {        // warp-uniform trip count (match / shfl below)
        const int64_t j0 = jb + tid;
        int64_t r[MC_U];
#pragma unroll
        for (int u = 0; u < MC_U; ++u) {
            const int64_t j = j0 + (int64_t)u * MC_THREADS;
            r[u] = j < nnz ? __ldg(rows + j) : -1;
        }
#pragma unroll
        for (int u = 0; u < MC_U; ++u) {
            // one atomic per distinct row of the warp (same-address shared atomics serialise a full round trip each)
            const int rr = (r[u] >= 0 && r[u] < B) ? (int)r[u] : -1;
            const unsigned peers = __match_any_sync(0xffffffffu, rr);
            if (rr >= 0 && lane == __ffs(peers) - 1) atomicAdd(cnt + rr, __popc(peers));
        }
    }
    __syncthreads();
    // exclusive scan of cnt[0..B]: each thread owns a contiguous run of rows
    const int per = (B + 1 + MC_THREADS - 1) / MC_THREADS;
    const int r0 = tid * per, r1 = min(B + 1, r0 + per);
    int local = 0;
    for (int r = r0; r < r1; ++r) local += cnt[r];
    int incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wtot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int v = wtot[lane], sc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, sc, o);
            if (lane >= o) sc += u;
        }
        wtot[lane] = sc - v;                                         // exclusive warp offsets
    }
    __syncthreads();
    int run = wtot[wid] + incl - local;
    for (int r = r0; r < r1; ++r) {
        const int c = cnt[r];
        ptr[r] = run;
        cnt[r] = run;                                                // becomes the fill cursor
        run += c;
    }
    __syncthreads();
    for (int64_t jb = 0; jb < nnz; jb += (int64_t)MC_U * MC_THREADS) {
        const int64_t j0 = jb + tid;
        int64_t r[MC_U], c[MC_U];
#pragma unroll
        for (int u = 0; u < MC_U; ++u) {
            const int64_t j = j0 + (int64_t)u * MC_THREADS;
            r[u] = j < nnz ? __ldg(rows + j) : -1;
            c[u] = j < nnz ? __ldg(cols + j) : 0;
        }
#pragma unroll
        for (int u = 0; u < MC_U; ++u) {
            const int rr = (r[u] >= 0 && r[u] < B) ? (int)r[u] : -1;
            const unsigned peers = __match_any_sync(0xffffffffu, rr);
            const int leader = __ffs(peers) - 1;
            int base = 0;
            if (rr >= 0 && lane == leader) base = atomicAdd(cnt + rr, __popc(peers));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (rr >= 0) items[base + __popc(peers & ((1u << lane) - 1u))] = (int32_t)(c[u] - item_offset);   // order inside a row is free
        }
    }
}
// large batches / masks: global count, library scan, fill
__global__ void mask_count_kernel(int64_t nnz, const int64_t* __restrict__ rows, int64_t B, int32_t* __restrict__ counts) {
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < nnz && rows[j] >= 0 && rows[j] < B) atomicAdd(counts + rows[j], 1);
}
__global__ void mask_fill_kernel(int64_t nnz, const int64_t* __restrict__ rows, const int64_t* __restrict__ cols, int64_t B,
                                 int64_t item_offset, const int32_t* __restrict__ ptr, int32_t* __restrict__ cursor,
                                 int32_t* __restrict__ items) {
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= nnz || rows[j] < 0 || rows[j] >= B) return;
    const int pos = ptr[rows[j]] + atomicAdd(cursor + rows[j], 1);
    items[pos] = (int32_t)(cols[j] - item_offset);     // may fall outside [0, n_items): then it never matches
}

// One launch per row block for everything the passes need prepared: the sorted-mask CSR (first call only), the user
// operand + row norms, and the zeroing of the flags / slot counter.
__global__ void __launch_bounds__(256) cf_prep_kernel(int64_t mask_blocks, int64_t mask_nnz, const int64_t* __restrict__ mask_rows,
                                                      const int64_t* __restrict__ mask_cols, int B_all, int64_t item_offset,
                                                      int32_t* __restrict__ mptr, int32_t* __restrict__ mitems, int32_t* __restrict__ unsorted,
                                                      int64_t nb, const int64_t* __restrict__ users, const float* __restrict__ Ue, int64_t ldu,
                                                      int d, int KP, uint4* __restrict__ Upk, float* __restrict__ unorm, int64_t pack_threads,
                                                      uint32_t* __restrict__ zero, int64_t zero_words) {
    if ((int64_t)blockIdx.x < mask_blocks) {
        cf_mask_sorted_block(blockIdx.x, mask_nnz, mask_rows, mask_cols, B_all, item_offset, mptr, mitems, unsorted);
        return;
    }
    int64_t t = (blockIdx.x - mask_blocks) * (int64_t)blockDim.x + threadIdx.x;
    if (t < pack_threads) { cf_pack_one(t, nb, users, Ue, ldu, d, KP, nullptr, Upk, unorm, nullptr); return; }   // (multiple of 256: whole blocks)
    t -= pack_threads;
    if (t < zero_words) zero[t] = 0;
}

// ------------------------------------------------------------------------------------------------------------------
// threshold: the need-th largest group maximum of the row, minus the certified margin.  One warp per row.
// ------------------------------------------------------------------------------------------------------------------
// Warp radix select over 32-bit keys read through `key_at(t)`, t < n: returns the key of the `need`-th largest.
template <typename F>
__device__ __forceinline__ uint32_t cf_warp_kth(F key_at, int n, int need, uint32_t* hist, int lane) {
    uint32_t prefix = 0;
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        const uint32_t hi_mask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
        for (int b = lane; b < 256; b += 32) hist[b] = 0;
        __syncwarp();
        for (int t = lane; t < n; t += 32) {
            const uint32_t key = key_at(t);
            if ((key & hi_mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
        }
        __syncwarp();
        // lane l owns bins [8l, 8l+8); `cum` = keys in the bins above (exclusive suffix sum)
        uint32_t mine[8], tot = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { mine[j] = hist[lane * 8 + j]; tot += mine[j]; }
        uint32_t incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_down_sync(0xffffffffu, incl, o);
            if (lane + o < 32) incl += v;
        }
        uint32_t cum = incl - tot;
        int dgt = -1;
#pragma unroll
        for (int j = 7; j >= 0; --j) {
            if (dgt < 0) {
                if (cum + mine[j] >= (uint32_t)need) dgt = lane * 8 + j;
                else cum += mine[j];
            }
        }
        const unsigned found = __ballot_sync(0xffffffffu, dgt >= 0);   // (never empty: need <= n)
        const int win = found ? 31 - __clz(found) : 0;
        dgt = __shfl_sync(0xffffffffu, dgt, win);
        cum = __shfl_sync(0xffffffffu, cum, win);
        if (dgt < 0) dgt = 0;
        prefix |= (uint32_t)dgt << shift;
        need -= (int)cum;
        __syncwarp();
    }
    return prefix;
}

// The threshold does not have to be the exact need-th largest group maximum -- any value with at least `need` maxima at
// or above it is certified.  So the search runs on the top CF_THR_BITS bits of the order-preserving key only (bit by
// bit, counts by REDUX: no atomics, the values stay in registers) and takes the lower edge of that bucket: 16 bits =
// the value to 2^-7 relative, a handful of extra candidates per row for half the dependent steps.
constexpr int CF_THR_BITS = 16;
template <int NV>
__device__ __forceinline__ uint32_t cf_warp_kth_coarse(const float* __restrict__ g, int G, int need, int lane) {
    uint32_t key[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int t = j * 32 + lane;
        key[j] = t < G ? float_key(__ldg(g + t)) : 0u;
    }
    // bits above the first one in which the row's largest and smallest key differ are common to all keys: nothing to search
    uint32_t kmax = 0u, kmin = 0xffffffffu;
#pragma unroll
    for (int j = 0; j < NV; ++j) {                                   // (-inf = a group of padding columns: not part of the range)
        kmax = max(kmax, key[j]);
        if (j * 32 + lane < G && key[j] > 0x007fffffu) kmin = min(kmin, key[j]);
    }
    kmax = __reduce_max_sync(0xffffffffu, kmax);
    kmin = __reduce_min_sync(0xffffffffu, kmin);
    const int top = 31 - __clz((kmax ^ kmin) | (1u << (32 - CF_THR_BITS)));    // >= the lowest searched bit
    uint32_t prefix = top >= 31 ? 0u : (kmax & ~((2u << top) - 1u));
#pragma unroll 1
    for (int b = top; b >= 32 - CF_THR_BITS; --b) {
        const uint32_t cand = prefix | (1u << b);
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < NV; ++j) cnt += key[j] >= cand;
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (cnt >= need) prefix = cand;
    }
    return prefix;                                                   // <= the need-th largest key, same top bits
}

__global__ void __launch_bounds__(256) cf_thr_kernel(int64_t nb, int G, int G_valid, int k, int d, const float* __restrict__ gmax, const float* __restrict__ unorm,
                                                     const uint32_t* __restrict__ max_norm, const int32_t* __restrict__ mask_ptr,
                                                     float* __restrict__ thr, int32_t* __restrict__ flags) {
    __shared__ uint32_t hist_all[8][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row = (int64_t)blockIdx.x * 8 + warp;
    if (row >= nb) return;
    const int need = k + (mask_ptr ? mask_ptr[row + 1] - mask_ptr[row] : 0);
    if (need > G_valid) {                                            // more finalists wanted than there are (non-padding) groups: exact kernel
        if (lane == 0) { thr[row] = INFINITY; flags[row] = 1; }
        return;
    }
    const float* g = gmax + row * G;
    uint32_t kth;
    if (G <= 16 * 32) kth = cf_warp_kth_coarse<16>(g, G, need, lane);
    else if (G <= 32 * 32) kth = cf_warp_kth_coarse<32>(g, G, need, lane);
    else kth = cf_warp_kth([&](int t) { return float_key(__ldg(g + t)); }, G, need, hist_all[warp], lane);
    if (lane == 0) {
        const float t = key_float(kth);
        // scaled domain.  Per element |dx| <= 2^-11 |x| + 2^-25 (fp16 subnormals), so
        //   |s~ - s| <= 2^-10 |u| |i| (1 + 2^-12) + 2^-25 sqrt(d) (|u| + |i|) + (2^-25)^2 d + accumulation  <=  eps' below;
        // with the largest elements scaled into [2^14, 2^15) the second term is ~2^-38 of the first
        const float un = unorm[row], mn = __uint_as_float(*max_norm);
        const float margin = 2.0f * (CF_EPS * un * mn + CF_EPS_SUB * sqrtf((float)d) * (un + mn + 1.0f));
        const float out = t - margin;
        if (!(fabsf(t) < INFINITY) || !(margin < INFINITY)) { thr[row] = INFINITY; flags[row] = 2; }   // NaN / inf scores
        else thr[row] = out;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// exact fp32 score of one (user, item) pair.  THE arithmetic of this file's results, chosen so that a group of lanes can
// compute it from one coalesced read of the item row:
//     L = 8 / 16 / 32 blocks of four elements (d <= 32 / 64 / 128; elements beyond d count as 0),
//     p_l = fmaf(u[4l+3], v[4l+3], fmaf(u[4l+2], v[4l+2], fmaf(u[4l+1], v[4l+1], fmaf(u[4l], v[4l], 0)))),
//     then the butterfly tree  p_a += p_(a + w)  for a < w,  w = L/2, L/4, ..., 1;  the score is p_0.
// cf_dot_thread is one thread doing all of it (exact kernel: every item of a flagged row); cf_dot_round is a warp doing
// 32 candidates, L lanes per item row, the tree run as a transposed butterfly so that each lane ends up with the
// complete score of one candidate.  Float addition commutes, so both give the same bits.
// ------------------------------------------------------------------------------------------------------------------
__host__ __device__ constexpr int cf_lpr(int d) { return d <= 32 ? 8 : (d <= 64 ? 16 : 32); }

__device__ __forceinline__ float4 cf_load4(const float* __restrict__ row, int l, int d, bool vec_ok) {
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec_ok) {                                                    // d % 4 == 0, rows 16-byte aligned
        if (4 * l < d) x = ldg4(row + 4 * l);
    } else {
        if (4 * l < d) x.x = __ldg(row + 4 * l);
        if (4 * l + 1 < d) x.y = __ldg(row + 4 * l + 1);
        if (4 * l + 2 < d) x.z = __ldg(row + 4 * l + 2);
        if (4 * l + 3 < d) x.w = __ldg(row + 4 * l + 3);
    }
    return x;
}
__device__ __forceinline__ float cf_chain4(const float4 u, const float4 x) {
    return fmaf(u.w, x.w, fmaf(u.z, x.z, fmaf(u.y, x.y, fmaf(u.x, x.x, 0.f))));
}

template <int LPR>
__device__ __forceinline__ float cf_dot_thread_t(const float* __restrict__ u_sm /* zero-padded to 128 */, const float* __restrict__ v, int d, bool vec_ok) {
    float p[LPR];
#pragma unroll
    for (int l0 = 0; l0 < LPR; l0 += 8) {                            // 8 x 16 bytes of the item row in flight
        float4 x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = cf_load4(v, l0 + i, d, vec_ok);
#pragma unroll
        for (int i = 0; i < 8; ++i) p[l0 + i] = cf_chain4(*reinterpret_cast<const float4*>(u_sm + 4 * (l0 + i)), x[i]);
    }
#pragma unroll
    for (int w = LPR / 2; w >= 1; w >>= 1)
#pragma unroll
        for (int a = 0; a < w; ++a) p[a] = p[a] + p[a + w];
    return p[0];
}
__device__ __forceinline__ float cf_dot_thread(const float* __restrict__ u_sm, const float* __restrict__ v, int d, bool vec_ok) {
    return d <= 32 ? cf_dot_thread_t<8>(u_sm, v, d, vec_ok) : (d <= 64 ? cf_dot_thread_t<16>(u_sm, v, d, vec_ok) : cf_dot_thread_t<32>(u_sm, v, d, vec_ok));
}

// 32 candidates cand[t0 .. t0 + 31] (negative = dropped, beyond n = absent): returns, in lane (sub, l) = (lane / LPR, lane % LPR),
// the score of candidate t0 + l * (32 / LPR) + sub.  `uu` = this lane's four elements 4l .. 4l + 3 of the user row.
// One load instruction covers 32 / LPR whole item rows (contiguous 16-byte pieces: every 128-byte line is touched once
// -- a lane per candidate touches 32 lines per instruction and the L1 tag stage becomes the limit).
template <int LPR>
__device__ __forceinline__ float cf_dot_round(const float4 uu, const float* __restrict__ Ie, int64_t ldi, int d, bool vec_ok,
                                              const int32_t* cand, int t0, int n, int lane) {
    constexpr int RPI = 32 / LPR, NI = LPR;
    const int l = lane & (LPR - 1), sub = lane / LPR;
    float p[NI];
#pragma unroll
    for (int h = 0; h < NI; h += 8) {
        float4 x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int t = t0 + (h + i) * RPI + sub;
            const int item = t < n ? cand[t] : -1;
            x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (item >= 0) x[i] = cf_load4(Ie + (int64_t)item * ldi, l, d, vec_ok);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) p[h + i] = cf_chain4(uu, x[i]);
    }
    // transposed butterfly: at width w the lanes with bit w set keep the upper half of their values, the others the lower
    // half, and each adds what its partner sends of the same candidates; value count and lane-group size halve together
#pragma unroll
    for (int w = LPR / 2; w >= 1; w >>= 1) {
        const bool up = (l & w) != 0;
#pragma unroll
        for (int a = 0; a < w; ++a) {
            const float keep = up ? p[a + w] : p[a];
            const float send = up ? p[a] : p[a + w];
            p[a] = keep + __shfl_xor_sync(0xffffffffu, send, w);
        }
    }
    return p[0];
}

// ------------------------------------------------------------------------------------------------------------------
// finalists: set bits of the row's bitmap -> unmasked -> exact fp32 -> top-k in contract order.  One warp per row, written
// for instruction count (the kernel is issue-bound at large batches: ~70 candidates per row, 20,000 rows):
//   * the set bits come out in ascending item order (lane = bitmap word, positions by a warp prefix sum);
//   * the mask is applied from the mask's side: lane q looks its masked item up in the sorted candidate list (binary
//     search), O(m log n) instead of n x m comparisons;
//   * exact scores 32 candidates at a time, 8 / 16 / 32 lanes per item row (cf_dot_round: coalesced reads);
//   * ranking counts, per element, the larger 32-bit value keys (one LDS broadcast feeds up to four elements of the
//     lane); equal values are ordered by item index = list position in a second pass that runs only when the rank sum
//     shows that two candidates share a value.
// ------------------------------------------------------------------------------------------------------------------
template <int E>
__device__ __forceinline__ void cf_rank_sweeps(const int32_t* cand, const uint32_t* keys, int n, int kept, int k, int lane, int64_t row,
                                               int64_t item_offset, int64_t* __restrict__ out_idx, float* __restrict__ out_val) {
    for (int e0 = 0; e0 * 32 < n; e0 += E) {
        uint32_t mk[E];
        int rk[E];
#pragma unroll
        for (int e = 0; e < E; ++e) { const int t = (e0 + e) * 32 + lane; mk[e] = t < n ? keys[t] : 0u; rk[e] = 0; }
        int u2 = 0;
        for (; u2 + 8 <= n; u2 += 8) {                               // 8 broadcast loads in flight, then the compares
            uint32_t ku[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) ku[i] = keys[u2 + i];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int e = 0; e < E; ++e) rk[e] += ku[i] > mk[e];
        }
        for (; u2 < n; ++u2) {
            const uint32_t ku = keys[u2];
#pragma unroll
            for (int e = 0; e < E; ++e) rk[e] += ku > mk[e];
        }
        // all value keys distinct <=> the ranks of the live elements are a permutation of 0 .. kept-1 (checkable when one
        // sweep covers the list; with several sweeps the tie pass always runs)
        bool tie = n > 32 * E;
        if (!tie) {
            int sr = 0;
#pragma unroll
            for (int e = 0; e < E; ++e) sr += mk[e] != 0u ? rk[e] : 0;
            tie = __reduce_add_sync(0xffffffffu, sr) != kept * (kept - 1) / 2;
        }
        if (tie) {                                                   // equal values: lower item index (= list position) first
            for (int u2 = 0; u2 < n; ++u2) {
                const uint32_t ku = keys[u2];
#pragma unroll
                for (int e = 0; e < E; ++e) rk[e] += (ku == mk[e]) && (u2 < (e0 + e) * 32 + lane);
            }
        }
#pragma unroll
        for (int e = 0; e < E; ++e) {
            if (mk[e] != 0u && rk[e] < k) {
                out_idx[row * k + rk[e]] = (int64_t)cand[(e0 + e) * 32 + lane] + item_offset;
                out_val[row * k + rk[e]] = key_float(mk[e]);
            }
        }
    }
}

constexpr int CF_FIN_WARPS = 4;
template <int LPR>
__global__ void __launch_bounds__(32 * CF_FIN_WARPS, LPR <= 16 ? 8 : 6) cf_final_kernel(int64_t nb, int n_it, int64_t n_items, int d, int k, int64_t item_offset,
                                                                     const uint4* __restrict__ bitmap, const int64_t* __restrict__ users,
                                                                     const float* __restrict__ Ue, int64_t ldu, const float* __restrict__ Ie, int64_t ldi,
                                                                     const int32_t* __restrict__ mask_ptr, const int32_t* __restrict__ mask_items,
                                                                     int32_t* __restrict__ flags, int32_t* __restrict__ counter,
                                                                     int32_t* __restrict__ row_of_slot, int64_t* __restrict__ out_idx,
                                                                     float* __restrict__ out_val) {
    __shared__ int32_t cand_all[CF_FIN_WARPS][CF_CAP];
    __shared__ uint32_t key_all[CF_FIN_WARPS][CF_CAP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row = (int64_t)blockIdx.x * CF_FIN_WARPS + warp;
    if (row >= nb) return;
    auto condemn = [&](int why) {                                    // the exact kernel takes the row
        if (lane == 0) {
            if (why) flags[row] = why;
            row_of_slot[atomicAdd(counter, 1)] = (int32_t)row;
        }
    };
    // everything that depends on the row number only is requested at once
    const int flagged = __ldg(flags + row);
    const int m0 = mask_ptr ? __ldg(mask_ptr + row) : 0, m1 = mask_ptr ? __ldg(mask_ptr + row + 1) : 0;
    const int64_t urow = users ? __ldg(users + row) : row;
    const uint4* bm = bitmap + row * n_it;
    uint4 b0 = make_uint4(0u, 0u, 0u, 0u);
    if (lane < n_it) b0 = __ldg(bm + lane);
    if (flagged) { condemn(0); return; }
    int32_t* cand = cand_all[warp];
    uint32_t* keys = key_all[warp];
    // 1. set bits -> candidate list in ascending item order; keys[] = 1 marks a live candidate
    int n = 0;
    for (int w0 = 0; w0 < n_it; w0 += 32) {
        const int wi = w0 + lane;
        uint4 b = b0;
        if (w0 > 0) { b = make_uint4(0u, 0u, 0u, 0u); if (wi < n_it) b = __ldg(bm + wi); }
        const int mine = __popc(b.x) + __popc(b.y) + __popc(b.z) + __popc(b.w);
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        int pos = n + incl - mine;
        n += __shfl_sync(0xffffffffu, incl, 31);
        if (mine) {
            const uint32_t ws[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t x = ws[q];
                while (x) {
                    const int j = __clz(x);                          // bit (31 - j) <-> column 32 q + j of the tile
                    x &= ~(0x80000000u >> j);
                    if (pos < CF_CAP) { cand[pos] = wi * CF_TILE + q * 32 + j; keys[pos] = 1u; }
                    ++pos;
                }
            }
        }
    }
    if (n > CF_CAP) { condemn(4); return; }
    __syncwarp();
    // 2. masked train positives out: each masked item is looked up in the sorted list, its key becomes 0 (= dropped)
    for (int q0 = m0; q0 < m1; q0 += 32) {
        const int q = q0 + lane;
        if (q < m1) {
            const int item = __ldg(mask_items + q);
            int lo = 0, hi = n;                                      // first position with cand >= item
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (cand[mid] < item) lo = mid + 1; else hi = mid;
            }
            if (lo < n && cand[lo] == item) keys[lo] = 0u;
        }
    }
    __syncwarp();
    // 3. exact fp32 scores (float_key of a real score is never 0; -NaN would be: such a candidate is dropped).  Dropped
    //    candidates are marked in cand[] first (sign bit) so that a round reads one word per candidate.
    for (int t = lane; t < n; t += 32)
        if (keys[t] == 0u || cand[t] >= n_items) cand[t] |= (int32_t)0x80000000;
    __syncwarp();
    const bool vec_ok = (ldi & 3) == 0 && (d & 3) == 0 && ((((uintptr_t)Ie) & 15) == 0);
    const bool vec_u = (ldu & 3) == 0 && (d & 3) == 0 && ((((uintptr_t)Ue) & 15) == 0);
    const float4 uu = cf_load4(Ue + urow * ldu, lane & (LPR - 1), d, vec_u);
    int kept = 0;
    for (int t0 = 0; t0 < n; t0 += 32) {
        const float sc = cf_dot_round<LPR>(uu, Ie, ldi, d, vec_ok, cand, t0, n, lane);
        const int t = t0 + (lane & (LPR - 1)) * (32 / LPR) + lane / LPR;
        if (t < n) {
            const uint32_t key = cand[t] >= 0 ? float_key(sc) : 0u;
            kept += key != 0u;
            keys[t] = key;
        }
    }
    kept = __reduce_add_sync(0xffffffffu, kept);
    __syncwarp();
    if (kept < k) { condemn(8); return; }                            // (cannot happen for finite scores: the threshold is certified)
    // 4. rank = number of candidates with a larger value key; E elements of this lane per sweep of the list
    if (n <= 64) cf_rank_sweeps<2>(cand, keys, n, kept, k, lane, row, item_offset, out_idx, out_val);
    else if (n <= 96) cf_rank_sweeps<3>(cand, keys, n, kept, k, lane, row, item_offset, out_idx, out_val);
    else cf_rank_sweeps<4>(cand, keys, n, kept, k, lane, row, item_offset, out_idx, out_val);
}

// ------------------------------------------------------------------------------------------------------------------
// exact fp32 rows (flagged only): all items on CUDA cores, mask, radix select, ordered ties, sort -- the contract of
// mmrec_topk_rows_f32.  CTA `sl` serves the flagged rows sl, sl + CF_EX_SLOTS, ... with its own key buffer; all CTAs
// exit at once when nothing was flagged.
// ------------------------------------------------------------------------------------------------------------------
__device__ void cf_bitonic_desc(uint64_t* a, int n) {
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
                int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                bool desc = ((lo & size) == 0);
                uint64_t x = a[lo], y = a[hi];
                if ((x < y) == desc) { a[lo] = y; a[hi] = x; }
            }
        }
    __syncthreads();
}

__global__ void __launch_bounds__(256) cf_exact_kernel(const int64_t* __restrict__ users, const float* __restrict__ Ue, int64_t ldu,
                                                       int64_t n_items, const float* __restrict__ Ie, int64_t ldi, int d, int k,
                                                       int64_t item_offset, const int32_t* __restrict__ mask_ptr,
                                                       const int32_t* __restrict__ mask_items, const int32_t* __restrict__ counter,
                                                       const int32_t* __restrict__ row_of_slot, unsigned* __restrict__ keys_all,
                                                       int64_t* __restrict__ out_idx, float* __restrict__ out_val) {
    __shared__ unsigned hist[256];
    __shared__ uint64_t sel[1024];
    __shared__ unsigned tie_idx[1024];
    __shared__ unsigned s_prefix, s_need, s_count, s_base, n_ties;
    __shared__ unsigned warp_tot[8];
    __shared__ __align__(16) float u_ex[128];
    const int n_flagged = *counter;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    unsigned* keys = keys_all + (int64_t)blockIdx.x * n_items;
    for (int fr = blockIdx.x; fr < n_flagged; fr += gridDim.x) {
        const int64_t row = row_of_slot[fr];
        __syncthreads();
        // ---- keys: one thread per item, cf_dot_thread's arithmetic (the row gets the same bits whichever kernel served it)
        const float* u = Ue + (users ? users[row] : row) * ldu;
        if (tid < 128) u_ex[tid] = tid < d ? u[tid] : 0.f;
        __syncthreads();
        const bool vec_ok = (ldi & 3) == 0 && (d & 3) == 0 && ((((uintptr_t)Ie) & 15) == 0);
        for (int64_t i = tid; i < n_items; i += 256) keys[i] = float_key(cf_dot_thread(u_ex, Ie + i * ldi, d, vec_ok));
        __syncthreads();
        const int m0 = mask_ptr ? mask_ptr[row] : 0, m1 = mask_ptr ? mask_ptr[row + 1] : 0;
        for (int q = m0 + tid; q < m1; q += 256) {
            const int64_t item = mask_items[q];
            if (item >= 0 && item < n_items) keys[item] = float_key(-1e10f);          // src/common/trainer.py:307
        }
        __syncthreads();
        // ---- radix select of the k-th largest key
        unsigned prefix = 0, need = (unsigned)k;
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            const unsigned hi_mask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
            hist[tid] = 0;
            __syncthreads();
            for (int64_t i = tid; i < n_items; i += 256) {
                const unsigned key = keys[i];
                if ((key & hi_mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (tid == 0) {
                unsigned cum = 0;
                int dgt = 255;
                for (; dgt > 0; --dgt) {
                    if (cum + hist[dgt] >= need) break;
                    cum += hist[dgt];
                }
                s_prefix = prefix | ((unsigned)dgt << shift);
                s_need = need - cum;
            }
            __syncthreads();
            prefix = s_prefix; need = s_need;
            __syncthreads();
        }
        const unsigned kth = prefix;
        if (tid == 0) { s_count = 0; s_base = 0; n_ties = 0; }
        __syncthreads();
        const unsigned n_gt = (unsigned)k - need;
        // strictly greater keys in any order; the indices of the keys equal to the k-th are collected and the `need` lowest
        // of them taken (normally there is exactly one)
        for (int64_t i = tid; i < n_items; i += 256) {
            const unsigned key = keys[i];
            if (key > kth) { unsigned pos = atomicAdd(&s_count, 1u); sel[pos] = ((uint64_t)key << 32) | (uint32_t)(~(uint32_t)i); }
            else if (key == kth) { unsigned pos = atomicAdd(&n_ties, 1u); if (pos < 1024u) tie_idx[pos] = (unsigned)i; }
        }
        __syncthreads();
        if (n_ties <= 1024u) {
            const unsigned nt = n_ties;
            for (unsigned t = tid; t < nt; t += 256) {
                const unsigned me = tie_idx[t];
                unsigned rank = 0;
                for (unsigned u2 = 0; u2 < nt; ++u2) rank += tie_idx[u2] < me;
                if (rank < need) sel[n_gt + rank] = ((uint64_t)kth << 32) | (uint32_t)(~me);
            }
        } else {
            // degenerate row (thousands of equal scores): ordered sweep, 256 items at a time
            for (int64_t i0 = 0; i0 < n_items; i0 += 256) {
                const int64_t i = i0 + tid;
                const bool eq = i < n_items && keys[i] == kth;
                const unsigned bal = __ballot_sync(0xffffffffu, eq);
                if (lane == 0) warp_tot[wid] = __popc(bal);
                __syncthreads();
                unsigned off = s_base;
                for (int w = 0; w < wid; ++w) off += warp_tot[w];
                const unsigned rank = off + __popc(bal & ((1u << lane) - 1u));
                if (eq && rank < need) sel[n_gt + rank] = ((uint64_t)kth << 32) | (uint32_t)(~(uint32_t)i);
                __syncthreads();
                if (tid == 0) { unsigned tot = 0; for (int w = 0; w < 8; ++w) tot += warp_tot[w]; s_base += tot; }
                __syncthreads();
                if (s_base >= need) break;
            }
        }
        __syncthreads();
        int n2 = 1;
        while (n2 < k) n2 <<= 1;
        for (int t = k + tid; t < n2; t += 256) sel[t] = 0;
        cf_bitonic_desc(sel, n2);
        for (int t = tid; t < k; t += 256) {
            const uint64_t c = sel[t];
            out_idx[row * k + t] = (int64_t)(uint32_t)(~(uint32_t)c) + item_offset;
            out_val[row * k + t] = key_float((uint32_t)(c >> 32));
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
static inline int cf_kp(int d) { return d <= 32 ? 32 : (d <= 64 ? 64 : 128); }
static inline int cf_gw(int64_t n_items) { return n_items <= 16384 ? 1 : (n_items <= 32768 ? 2 : (n_items <= 65536 ? 4 : 8)); }

constexpr size_t CF_CAT_HEADER = 1024;          // {max scaled item norm (fp32 bits), n_items, d, KP, largest |element| (fp32 bits)} + padding

size_t cf_catalog_bytes(int64_t n_items, int d) {
    if (n_items <= 0 || d < 1 || d > 128) return 0;
    const int64_t n_it = (n_items + CF_TILE - 1) / CF_TILE;
    return CF_CAT_HEADER + (size_t)n_it * CF_TILE * cf_kp(d) * 2;
}

int cf_catalog_pack(int64_t n_items, const float* Ie, int64_t ldi, int d, void* cat, size_t cat_bytes, cudaStream_t stream) {
    const size_t need = cf_catalog_bytes(n_items, d);
    if (!need || !cat || cat_bytes < need || (((uintptr_t)cat) & 1023)) { set_error("catalog_pack: bad shape, or buffer null / not 1024-byte aligned / smaller than mmrec_catalog_bytes"); return MMREC_EINVAL; }
    const int KP = cf_kp(d);
    const int64_t n_it = (n_items + CF_TILE - 1) / CF_TILE;
    MMREC_CUDA(cudaMemsetAsync(cat, 0, CF_CAT_HEADER, stream));
    {
        const int64_t blocks = (n_items + 7) / 8;
        cf_item_absmax_kernel<<<(unsigned)(blocks < 2368 ? blocks : 2368), 256, 0, stream>>>(n_items, Ie, ldi, d, (uint32_t*)cat);
        MMREC_LAUNCH_CHECK();
    }
    const int64_t threads = n_it * CF_TILE * (KP / 8);
    cf_pack_items_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(n_items, Ie, ldi, d, KP, (uint4*)((char*)cat + CF_CAT_HEADER),
                                                                                  (uint32_t*)cat, threads);
    MMREC_LAUNCH_CHECK();
    return MMREC_OK;
}

struct CfPlan {
    int KP, gw, G;
    int64_t n_it, rows_blk, rows_pad, n_pairs;
    size_t off_cat, off_upk, off_unorm, off_gmax, off_thr, off_bitmap, off_flags, off_mptr, off_mcur, off_mitems, off_cub, off_keys, cub_bytes, total;
};

static CfPlan cf_plan(int64_t B, int64_t n_items, int d, int64_t mask_nnz, bool with_cat) {
    CfPlan P;
    P.KP = cf_kp(d);
    P.gw = cf_gw(n_items);
    P.n_it = (n_items + CF_TILE - 1) / CF_TILE;
    P.G = (int)(P.n_it * (8 / P.gw));
    // row block: group maxima + bitmap of a block stay below ~512 MB
    const int64_t per_row = (int64_t)P.G * 4 + P.n_it * 16;
    int64_t rb = (512ll << 20) / per_row / (2 * CF_TILE) * (2 * CF_TILE);
    if (rb < 2 * CF_TILE) rb = 2 * CF_TILE;
    if (rb > 65536) rb = 65536;
    P.rows_blk = B < rb ? B : rb;
    P.rows_pad = (P.rows_blk + 2 * CF_TILE - 1) / (2 * CF_TILE) * (2 * CF_TILE);
    P.n_pairs = P.rows_pad / (2 * CF_TILE);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 1024); return o; };
    P.off_cat = take(with_cat ? cf_catalog_bytes(n_items, d) : 0);
    P.off_upk = take((size_t)P.rows_pad * P.KP * 2);
    P.off_unorm = take((size_t)P.rows_pad * 4);
    P.off_gmax = take((size_t)P.rows_blk * P.G * 4);
    P.off_thr = take((size_t)P.rows_pad * 4);
    P.off_bitmap = take((size_t)P.rows_blk * P.n_it * 16);
    P.off_flags = take((size_t)(2 * P.rows_blk + 2) * 4);            // flags [rows_blk] | counter | row_of_slot [rows_blk]   (flags + counter zeroed per block)
    P.off_mptr = take((size_t)(B + 2) * 4);
    P.off_mcur = take((size_t)(B + 2 > 1100 ? B + 2 : 1100) * 4);    // fill cursors, or the per-block order flags of the sorted-mask pass
    P.off_mitems = take((size_t)(mask_nnz > 0 ? mask_nnz : 1) * 4);
    size_t scan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (int32_t*)nullptr, (int32_t*)nullptr, (int64_t)(B + 1));
    P.cub_bytes = scan_bytes;
    P.off_cub = take(scan_bytes);
    P.off_keys = take((size_t)CF_EX_SLOTS * n_items * 4);
    P.total = off + 1024;
    return P;
}

bool score_cf_supported(int64_t B, int64_t n_items, int d, int k) {
    if (!(B > 0 && d >= 1 && d <= 128 && k >= 1 && k <= 256 && n_items < (1ll << 31))) return false;
    const int64_t G = (n_items + CF_TILE - 1) / CF_TILE * (8 / cf_gw(n_items));
    return G >= 2 * (int64_t)k;                                      // enough groups for need = k + masked items (rows that want more go to the exact kernel)
}

size_t score_cf_workspace_bytes(int64_t B, int64_t n_items, int d, int k, int64_t mask_nnz, bool with_cat) {
    if (!score_cf_supported(B, n_items, d, k)) return 0;
    return cf_plan(B, n_items, d, mask_nnz, with_cat).total;
}

static int cf_set_attrs() {
    static bool done[64] = {false};
    int dev = 0;
    MMREC_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !done[dev]) {                        // the attribute is per device
        MMREC_CUDA(cudaFuncSetAttribute(cf_pass_kernel<1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        MMREC_CUDA(cudaFuncSetAttribute(cf_pass_kernel<1, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        MMREC_CUDA(cudaFuncSetAttribute(cf_pass_kernel<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        MMREC_CUDA(cudaFuncSetAttribute(cf_pass_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        MMREC_CUDA(cudaFuncSetAttribute(cf_pass_kernel<2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        MMREC_CUDA(cudaFuncSetAttribute(mask_csr_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        if (dev >= 0 && dev < 64) done[dev] = true;
    }
    return MMREC_OK;
}

// Stage timing (tuning aid): with env MMREC_CF_TIMING set, the stages of the LAST score_cf call are bracketed by CUDA events
// (not under stream capture); mmrec_debug_cf_timing reads them back in microseconds.
static cudaEvent_t g_cf_ev[10];
static int g_cf_nev = 0, g_cf_timing = -1;
static inline void cf_mark(cudaStream_t stream) {
    if (g_cf_timing <= 0 || g_cf_nev >= 10) return;
    if (!g_cf_ev[g_cf_nev]) cudaEventCreate(&g_cf_ev[g_cf_nev]);
    cudaEventRecord(g_cf_ev[g_cf_nev++], stream);
}
int score_cf_timing(float* us, int cap) {
    int n = 0;
    for (int i = 0; i + 1 < g_cf_nev && n < cap; ++i) {
        cudaEventSynchronize(g_cf_ev[i + 1]);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, g_cf_ev[i], g_cf_ev[i + 1]);
        us[n++] = ms * 1000.f;
    }
    return n;
}

// returns 1 = done, 0 = unsupported shape / workspace (caller uses the unfused path), <0 error.  `cat` = a catalogue packed
// by cf_catalog_pack for exactly (n_items, Ie, d), or NULL: then it is packed into the workspace first.
int score_cf(int64_t B, const int64_t* users, const float* Ue, int64_t ldu, int64_t n_items, const float* Ie, int64_t ldi,
             int d, const void* cat, int64_t mask_nnz, const int64_t* mask_rows, const int64_t* mask_cols, int k, int64_t item_offset,
             int64_t* out_idx, float* out_val, void* ws, size_t ws_bytes, cudaStream_t stream) {
    if (!score_cf_supported(B, n_items, d, k) || !ws) return 0;
    const CfPlan P = cf_plan(B, n_items, d, mask_nnz, cat == nullptr);
    char* base = (char*)(((uintptr_t)ws + 1023) & ~(uintptr_t)1023);
    if (ws_bytes < P.total + (size_t)(base - (char*)ws)) return 0;
    { int rc = cf_set_attrs(); if (rc) return rc; }
    if (g_cf_timing < 0) g_cf_timing = getenv("MMREC_CF_TIMING") ? 1 : 0;
    g_cf_nev = 0;
    cf_mark(stream);                                                  // stages: pack | prep + mask | pass 1 | thr | pass 2 | final | exact
    if (!cat) {
        int rc = cf_catalog_pack(n_items, Ie, ldi, d, base + P.off_cat, cf_catalog_bytes(n_items, d), stream);
        if (rc) return rc;
        cat = base + P.off_cat;
    }
    cf_mark(stream);
    const uint32_t* max_norm = (const uint32_t*)cat;
    const char* Ipk = (const char*)cat + CF_CAT_HEADER;
    uint4* Upk = (uint4*)(base + P.off_upk);
    float *unorm = (float*)(base + P.off_unorm), *gmax = (float*)(base + P.off_gmax), *thr = (float*)(base + P.off_thr);
    uint4* bitmap = (uint4*)(base + P.off_bitmap);
    int32_t* flags = (int32_t*)(base + P.off_flags);
    int32_t* counter = flags + P.rows_blk;
    int32_t* row_of_slot = counter + 1;
    int32_t *mptr = (int32_t*)(base + P.off_mptr), *mcur = (int32_t*)(base + P.off_mcur), *mitems = (int32_t*)(base + P.off_mitems);
    unsigned* keys = (unsigned*)(base + P.off_keys);
    const int T = 256;
    const bool has_mask = mask_nnz > 0;
    const bool small_mask = has_mask && B <= MC_MAX_ROWS && mask_nnz <= (1ll << 18);
    if (has_mask && !small_mask) {
        MMREC_CUDA(cudaMemsetAsync(mcur, 0, (size_t)(B + 2) * 4, stream));
        mask_count_kernel<<<(unsigned)((mask_nnz + T - 1) / T), T, 0, stream>>>(mask_nnz, mask_rows, B, mcur);
        MMREC_LAUNCH_CHECK();
        size_t tmp = P.cub_bytes;
        MMREC_CUDA(cub::DeviceScan::ExclusiveSum(base + P.off_cub, tmp, mcur, mptr, B + 1, stream));
        MMREC_CUDA(cudaMemsetAsync(mcur, 0, (size_t)(B + 2) * 4, stream));
        mask_fill_kernel<<<(unsigned)((mask_nnz + T - 1) / T), T, 0, stream>>>(mask_nnz, mask_rows, mask_cols, B, item_offset, mptr, mcur, mitems);
        MMREC_LAUNCH_CHECK();
    }
    const CfSmem L = cf_smem(P.KP);
    const int sms = sm_count();
    for (int64_t r0 = 0; r0 < B; r0 += P.rows_blk) {
        const int64_t nb = (B - r0) < P.rows_blk ? (B - r0) : P.rows_blk;
        const int64_t nb_pad = (nb + 2 * CF_TILE - 1) / (2 * CF_TILE) * (2 * CF_TILE);
        const int64_t n_pairs = nb_pad / (2 * CF_TILE);
        const int64_t* ub = users ? users + r0 : nullptr;
        const float* ue = users ? Ue : Ue + r0 * ldu;
        const int32_t* mp = has_mask ? mptr + r0 : nullptr;
        // prep: [mask CSR of the whole batch (first block, sorted case)] + user operand + zeroed flags / counter
        const int64_t mask_blocks = (small_mask && r0 == 0) ? (mask_nnz + 1 + T - 1) / T : 0;      // <= 1025 words of mcur hold the order flags
        const int64_t pack_threads = nb_pad * (P.KP / 8);
        const int64_t zero_words = P.rows_blk + 1;
        cf_prep_kernel<<<(unsigned)(mask_blocks + (pack_threads + zero_words + T - 1) / T), T, 0, stream>>>(
            mask_blocks, mask_nnz, mask_rows, mask_cols, (int)B, item_offset, mptr, mitems, mcur, nb, ub, ue, ldu, d, P.KP, Upk, unorm,
            pack_threads, (uint32_t*)flags, zero_words);
        MMREC_LAUNCH_CHECK();
        if (mask_blocks) {
            mask_csr_small_kernel<<<1, MC_THREADS, (size_t)(B + 1 + 32) * 4, stream>>>(mask_nnz, mask_rows, mask_cols, (int)B, item_offset, mptr,
                                                                                     mitems, mcur, (int)mask_blocks);
            MMREC_LAUNCH_CHECK();
        }
        cf_mark(stream);
        CfParams p;
        p.Upk = (const char*)Upk; p.Ipk = Ipk; p.KP = P.KP; p.n_it = (int)P.n_it; p.B = nb; p.n_items = n_items; p.n_units = n_pairs * P.n_it;
        p.gmax = gmax; p.G = P.G; p.gw = P.gw; p.thr = thr; p.bitmap = bitmap;
        { static int dbg = -1; if (dbg < 0) { const char* e = getenv("MMREC_CF_DEBUG"); dbg = e ? atoi(e) : 0; } p.dbg = dbg; }
        const unsigned grid = (unsigned)(p.n_units < sms ? p.n_units : sms);
        switch (P.gw) {
            case 1: cf_pass_kernel<1, 8><<<grid, CF_THREADS, L.total, stream>>>(p); break;
            case 2: cf_pass_kernel<1, 4><<<grid, CF_THREADS, L.total, stream>>>(p); break;
            case 4: cf_pass_kernel<1, 2><<<grid, CF_THREADS, L.total, stream>>>(p); break;
            default: cf_pass_kernel<1, 1><<<grid, CF_THREADS, L.total, stream>>>(p); break;
        }
        MMREC_LAUNCH_CHECK();
        cf_mark(stream);
        cf_thr_kernel<<<(unsigned)((nb + 7) / 8), 256, 0, stream>>>(nb, P.G, (int)((n_items + 16 * P.gw - 1) / (16 * P.gw)), k, d, gmax, unorm, max_norm, mp, thr, flags);
        MMREC_LAUNCH_CHECK();
        cf_mark(stream);
        cf_pass_kernel<2, 8><<<grid, CF_THREADS, L.total, stream>>>(p);
        MMREC_LAUNCH_CHECK();
        cf_mark(stream);
        {
            const unsigned fg = (unsigned)((nb + CF_FIN_WARPS - 1) / CF_FIN_WARPS);
#define CF_FINAL(LPR) cf_final_kernel<LPR><<<fg, 32 * CF_FIN_WARPS, 0, stream>>>(nb, (int)P.n_it, n_items, d, k, item_offset, bitmap, ub, ue, ldu, Ie, ldi, mp, \
                                                                            mitems, flags, counter, row_of_slot, out_idx + r0 * k, out_val + r0 * k)
            if (cf_lpr(d) == 8) CF_FINAL(8); else if (cf_lpr(d) == 16) CF_FINAL(16); else CF_FINAL(32);
#undef CF_FINAL
        }
        MMREC_LAUNCH_CHECK();
        cf_mark(stream);
        cf_exact_kernel<<<CF_EX_SLOTS, 256, 0, stream>>>(ub, ue, ldu, n_items, Ie, ldi, d, k, item_offset, mp, mitems, counter, row_of_slot, keys,
                                                         out_idx + r0 * k, out_val + r0 * k);
        MMREC_LAUNCH_CHECK();
        cf_mark(stream);
    }
    return 1;
}

// rows of the last row block that went to the exact kernel (synchronises; diagnostic)
int64_t score_cf_fallback_rows(const void* ws, int64_t B, int64_t n_items, int d, int k, int64_t mask_nnz, bool with_cat) {
    if (!score_cf_supported(B, n_items, d, k) || !ws) return -1;
    const CfPlan P = cf_plan(B, n_items, d, mask_nnz, with_cat);
    const char* base = (const char*)(((uintptr_t)ws + 1023) & ~(uintptr_t)1023);
    int32_t n = 0;
    if (cudaMemcpy(&n, base + P.off_flags + (size_t)P.rows_blk * 4, 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    if (getenv("MMREC_DEBUG")) {
        const int64_t nb = B % P.rows_blk ? B % P.rows_blk : P.rows_blk;
        int32_t* h = (int32_t*)malloc((size_t)nb * 4);
        if (h && cudaMemcpy(h, base + P.off_flags, (size_t)nb * 4, cudaMemcpyDeviceToHost) == cudaSuccess) {
            long long why[4] = {0, 0, 0, 0};
            for (int64_t i = 0; i < nb; ++i)
                for (int b = 0; b < 4; ++b) why[b] += (h[i] >> b) & 1;
            fprintf(stderr, "mmrec: exact-path rows %d of %lld (need > groups %lld, non-finite %lld, > %d candidates %lld, < k kept %lld)\n", n,
                    (long long)nb, why[0], why[1], CF_CAP, why[2], why[3]);
        }
        free(h);
    }
    return n;
}

}  // namespace mmrec
