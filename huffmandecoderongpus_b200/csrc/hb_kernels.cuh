/*
 * hb_kernels.cuh -- the sm_100a decode kernels.
 *
 * Functional phases (reference naming in brackets, SURVEY.md D4):
 *   hb_sync_kernel   phase 1+2 inside a tile: every thread decodes the chain of
 *                    codewords through its own subsequence, neighbouring chains
 *                    are stitched until all entry offsets agree, and the tile's
 *                    entry-offset -> (exit offset, symbol count) map is formed
 *                    [decodeAllBits + makebigtable, fastgpu.cu:46-93, but one
 *                    probe per CODEWORD of a handful of chains instead of one
 *                    tree walk per BIT plus log2(n) full-array passes]
 *   hb_scan_*        composition of the tile maps across the stream: exact
 *                    entry offset and output base of every tile
 *                    [calcbitsindex's top-down index broadcast, fastgpu.cu:96-113]
 *   hb_emit_kernel   decode the now-known chains and write bytes through a
 *                    shared-memory staging buffer with 16-byte stores
 *                    [calcresult + findmax, fastgpu.cu:116-138]
 *
 * Data layout in HBM: the compressed stream as little-endian u32 words
 * (16-byte aligned); per subsequence one u16 record (entry offset | count<<5);
 * per tile one 32 x u32 map; per 32 tiles / per 1024 tiles one 32 x u64 map.
 */
#ifndef HB_KERNELS_CUH_
#define HB_KERNELS_CUH_

#include <cuda_runtime.h>
#include <stdint.h>
#include "hb_core.cuh"
#include "huffb200.h"

#define HB_T 256            /* threads per CTA = subsequences per tile */
#ifndef HB_SYNC_MIN_CTAS
#define HB_SYNC_MIN_CTAS 6  /* register budget of the sync kernel: 65536 / (6 * 256) = 42 */
#endif
#define HB_SCAN_T 1024      /* threads per CTA of the scan kernels (32 warps x 32 tiles) */

struct hb_stream_args {
    const uint32_t *words;   /* compressed stream */
    uint64_t nwords;         /* readable words */
    uint64_t bits_own;       /* codewords starting before this bit are ours */
    uint64_t bits_avail;     /* valid bits in words[] (>= bits_own) */
    uint32_t ntiles;
    const uint32_t *lut;     /* single-symbol multi-level LUT in global memory */
    uint32_t w1;             /* its level-1 width */
    uint32_t maxlen;         /* number of candidate entry offsets to resolve */
    uint32_t minlen;         /* == maxlen: fixed-length code, closed-form chains */
    const uint32_t *fast;    /* S-table (sync kernel) or E-table (emit kernel), 1 << wf entries */
    uint32_t wf;
    uint32_t gmod, gorg;     /* When every codeword length is a multiple of g, codeword starts stay in ONE
                              * residue class mod g of the stream's bit positions (the stream begins on a
                              * codeword).  A tile at bit position P of the stream can then only be entered
                              * at offsets e with (P + e) % g == 0; chains of other offsets never merge with
                              * the true one -- following them anyway (round 1) made such codes 18 to 100
                              * times slower.  gmod = g when the shard's position in the stream is known
                              * (hb_ctx_set_shard_origin; gorg = that position in bits mod g), else the
                              * largest power of two dividing g, which needs no position because shards,
                              * chunks and tiles all begin at multiples of 128 bits (gorg = 0). */
};

/* fast-table footprint in shared memory, kept a multiple of 16 bytes */
__host__ __device__ __forceinline__ uint32_t hb_lut_smem_words(uint32_t wf) {
    return ((1u << wf) + 3u) & ~3u;
}

/* Launder a shared-space address through an empty asm so that the compiler keeps
 * it in a register instead of re-deriving it (S2UR SR_CgaCtaId + ULEA) inside
 * the probe loops. */
__device__ __forceinline__ uint32_t hb_opaque(uint32_t v) {
    asm volatile("" : "+r"(v));
    return v;
}

/* may a chain enter tile `tile` (tile_bits bits per tile) at offset e?  (hb_stream_args.gmod) */
__device__ __forceinline__ bool hb_entry_possible(const hb_stream_args &a, uint32_t tile, uint32_t tile_bits,
                                                  uint32_t e) {
    if (a.gmod <= 1u) return true;
    const uint32_t p = (a.gorg + (tile % a.gmod) * (tile_bits % a.gmod) + e) % a.gmod;
    return p == 0u;
}

/* The first offset at which a chain can enter the subsequence that begins sub_bit0 bits into tile
 * `tile`: the guess the probe sync kernel starts from.  0 unless the code's lengths share a factor
 * that is not a power of two (hb_stream_args.gmod): subsequences are 32 * WPT bits long, so their
 * starts wander through the residue classes mod 3, 5, ... and the guess "a codeword starts at my
 * bit 0" would be in the wrong class most of the time -- chains of different classes never merge,
 * and the stitch then needs one round per subsequence of the tile (round 2: 5.5 GB/s). */
__device__ __forceinline__ uint32_t hb_first_entry(const hb_stream_args &a, uint32_t tile, uint32_t tile_bits,
                                                   uint32_t sub_bit0) {
    if (a.gmod <= 1u) return 0u;
    const uint32_t p = (a.gorg + (tile % a.gmod) * (tile_bits % a.gmod) + sub_bit0 % a.gmod) % a.gmod;
    return p ? a.gmod - p : 0u;
}

/* device status word bits */
#define HB_ST_OUTPUT_FULL 1u

/* EXTRA = false: w[WPT] (the first word of the next subsequence) is left to the caller -- a load of one
 * word per thread is 9 more tag lookups per warp on the pipe the sync kernel is bound by */
template <int WPT, bool EXTRA = true>
__device__ __forceinline__ void hb_load_words(const hb_stream_args &a, uint64_t wbase,
                                              uint32_t (&w)[WPT + 1]) {
    if (wbase + WPT + 1 <= a.nwords) {
        if (WPT % 8 == 0 && (reinterpret_cast<uintptr_t>(a.words) & 31u) == 0) {
            /* 32-byte aligned stream: one 256-bit load per 8 words (sm_100 LDG.256) -- a warp
             * then touches every 128-byte line once instead of twice */
#pragma unroll
            for (int v = 0; v < WPT / 8; v++)
                asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                             : "=r"(w[8 * v]), "=r"(w[8 * v + 1]), "=r"(w[8 * v + 2]), "=r"(w[8 * v + 3]),
                               "=r"(w[8 * v + 4]), "=r"(w[8 * v + 5]), "=r"(w[8 * v + 6]), "=r"(w[8 * v + 7])
                             : "l"(a.words + wbase + 8 * v));
        } else {
            const uint4 *p = reinterpret_cast<const uint4 *>(a.words + wbase);
#pragma unroll
            for (int v = 0; v < WPT / 4; v++) {
                uint4 q = __ldg(p + v);
                w[4 * v + 0] = q.x; w[4 * v + 1] = q.y; w[4 * v + 2] = q.z; w[4 * v + 3] = q.w;
            }
        }
        if (EXTRA) w[WPT] = __ldg(a.words + wbase + WPT);
    } else {
#pragma unroll
        for (int j = 0; j < WPT + (EXTRA ? 1 : 0); j++)
            w[j] = (wbase + j < a.nwords) ? __ldg(a.words + wbase + j) : 0u;
    }
}

/* exclusive block scan of one u32 per thread (HB_T threads); returns the prefix,
 * *total receives the block sum.  s_warp: >= 9 words of shared memory. */
__device__ __forceinline__ uint32_t hb_block_exscan(uint32_t v, uint32_t *s_warp,
                                                    uint32_t *total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += y;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t x = (lane < HB_T / 32) ? s_warp[lane] : 0u;
        uint32_t xi = x;
#pragma unroll
        for (int d = 1; d < HB_T / 32; d <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, xi, d);
            if (lane >= d) xi += y;
        }
        if (lane < HB_T / 32) s_warp[lane] = xi - x;
        if (lane == HB_T / 32 - 1) s_warp[HB_T / 32] = xi;
    }
    __syncthreads();
    uint32_t pre = s_warp[wid] + inc - v;
    *total = s_warp[HB_T / 32];
    return pre;
}

/* ------------------------------------------------------------------------- */
template <int WPT>
__global__ void __launch_bounds__(HB_T, HB_SYNC_MIN_CTAS)
hb_sync_kernel(hb_stream_args a, uint32_t tile0, uint16_t *__restrict__ subs, uint32_t *__restrict__ tmaps) {
    constexpr int T = HB_T;
    constexpr uint32_t S = 32u * WPT;
    constexpr uint32_t TS = T * S;
    __shared__ __align__(16) uint32_t s_fast[1u << HB_WF_MAX];   /* S-table (static: constant address) */
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t *s_comp = smem;                               /* T*WPT + 4 */
    uint32_t *s_rec = s_comp + T * WPT + 4;                /* WPT*T per-word (land, cnt) */
    uint32_t *s_cs = s_rec + WPT * T;                      /* T */
    uint32_t *s_land = s_cs + T;                           /* T: landing behind each subsequence */
    uint32_t *s_warp = s_land + T;                         /* 16 */
    const int t = threadIdx.x;

    for (uint32_t i = t; i < (1u << a.wf); i += T) s_fast[i] = __ldg(a.fast + i);
    __syncthreads();
    hb_tables tb;
    tb.fast = s_fast;
    tb.fast_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_fast));
    tb.fmask4 = ((1u << a.wf) - 1u) << 2;
    tb.slow = hb_lutref{a.lut, a.lut, (1u << a.w1) - 1u};

    const bool fixed_len = a.minlen == a.maxlen;
    for (uint32_t tile = tile0 + blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        const uint64_t tile_bit0 = (uint64_t)tile * TS;
        const uint64_t sub0 = tile_bit0 + (uint64_t)t * S;
        uint32_t w[WPT + 1];
        hb_load_words<WPT>(a, (uint64_t)tile * (T * WPT) + (uint64_t)t * WPT, w);
#pragma unroll
        for (int j = 0; j < WPT; j++) s_comp[t * WPT + j] = w[j];
        if (t == T - 1) s_comp[T * WPT] = w[WPT];

        const uint32_t lim = sub0 >= a.bits_own ? 0u
                           : (a.bits_own - sub0 < S ? (uint32_t)(a.bits_own - sub0) : S);

        /* chain of the guess "a codeword starts at offset 0 of my subsequence"
         * (for a fixed-length code the exact offset under tile entry 0 is known) */
        uint32_t rec[WPT];
        uint32_t e = fixed_len ? hb_fixed_next(0u, a.maxlen, (uint32_t)t * S) - (uint32_t)t * S
                               : hb_first_entry(a, tile, TS, (uint32_t)t * S);
        hb_walk<WPT>(tb, w, lim, e, rec);
        s_land[t] = hb_rec_land(rec[WPT - 1]);
        __syncthreads();

        /* stitch: my true entry is where my left neighbour's chain lands; repeat
         * until no landing moves (1-3 rounds on self-synchronising data, at most
         * T rounds in general) */
        for (;;) {
            bool changed = false;
            if (t > 0 && lim > 0) {
                const uint32_t en = s_land[t - 1];
                if (en != e) {
                    e = en;
                    changed = hb_rewalk<WPT>(tb, w, lim, e, rec);
                }
            }
            if (!__syncthreads_or(changed)) break;
            s_land[t] = hb_rec_land(rec[WPT - 1]);
            __syncthreads();
        }

        uint32_t c = 0;
#pragma unroll
        for (int j = 0; j < WPT; j++) {
            c += hb_rec_cnt(rec[j]);
            s_rec[j * T + t] = rec[j];
        }
        subs[(uint64_t)tile * T + t] = hb_sub_pack(e, c);

        uint32_t C0;
        uint32_t pre = hb_block_exscan(c, s_warp, &C0);
        s_cs[t] = pre;
        __syncthreads();

        /* tile map: hypothesis 0 is the converged chain; hypotheses 1..maxlen-1
         * are followed by one lane each until they land on it */
        if (t < 32) {
            const uint64_t own_left = a.bits_own - tile_bit0;   /* tile < ntiles => > 0 */
            const uint32_t tile_lim = own_left < TS ? (uint32_t)own_left : TS;
            const uint32_t wl = (tile_lim - 1u) >> 5;           /* last owned word */
            const uint32_t X0 = hb_rec_land(s_rec[(wl % WPT) * T + wl / WPT]);
            uint32_t m = hb_map_pack32(X0, C0);
            if (t > 0 && (uint32_t)t < a.maxlen && hb_entry_possible(a, tile, TS, (uint32_t)t)) {
                if (fixed_len) {   /* never merges: arithmetic progression t, t+len, ... */
                    const uint32_t n = hb_fixed_count((uint32_t)t, a.maxlen, 0u, tile_lim);
                    m = hb_map_pack32((hb_fixed_next((uint32_t)t, a.maxlen, tile_lim) - tile_lim) & 31u, n);
                } else {
                    m = hb_hyp_walk<WPT, T>(tb, s_comp, s_rec, s_cs, C0, X0, tile_lim, (uint32_t)t);
                }
            }
            tmaps[(uint64_t)tile * 32 + t] = m;
        }
        __syncthreads();
    }
}

/* ------------------------------------------------------------------------- */
/* Code tables built on the device from the node array (SURVEY 8(f) rank 1; the reference
 * has a dead precedent in framework/fastgpuOpt1.cu:22-49).  One thread per table entry:
 * entries [0, 1 << wf) are the three multi-symbol tables (same index, one walk of at most
 * wf bits), entries after that the transducer table (state, byte).  The host only
 * validates the tree, numbers the states and builds the small single-symbol table
 * (hb_lut_build_small); csrc/hb_lut.c keeps the full host construction as the reference
 * the tests compare this kernel against, entry by entry. */
struct hb_build_args {
    const hb_node_abi *tree;      /* reference node array, 12-byte structs */
    const int32_t *node_state;    /* state of every node, -1 for leaves */
    const int32_t *state_node;    /* node of every state */
    uint32_t nstates, wf, wf64;   /* wf64 <= wf: index width of the E64-table */
    uint32_t *stab, *etab, *e64;
    uint16_t *fsm;                /* NULL when the tree has no transducer */
};

__global__ void __launch_bounds__(256)
hb_build_tables_kernel(hb_build_args b) {
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    const uint32_t nf = 1u << b.wf;
    if (i < nf) {
        const uint32_t x = i;
        uint32_t sm = 0, nsym = 0, used = 0, syms = 0, pos = 0;
        uint32_t used2 = 0, used4 = 0, n4 = 0;   /* bits used by the first two codewords / by the first (at most four) that end within wf64 bits */
        for (;;) {
            int32_t node = 0;
            uint32_t p = pos;
            while (b.tree[node].izero != -1 && p < b.wf) {
                node = ((x >> p) & 1u) ? b.tree[node].ione : b.tree[node].izero;
                p++;
            }
            if (b.tree[node].izero != -1) break;      /* next codeword does not fit */
            sm |= 1u << pos;
            if (nsym < 4u) syms |= (uint32_t)b.tree[node].sym << (8u * nsym);
            nsym++;
            used = p;
            if (nsym <= 2u) used2 = p;
            if (nsym <= 4u && p <= b.wf64) { used4 = p; n4 = nsym; }
            pos = p;
            if (pos >= b.wf) break;
        }
        if (nsym == 0) {
            b.stab[x] = HB_FAST_MARK << 16;
            b.etab[x] = HB_FAST_MARK << 16;
        } else {
            const uint32_t n2 = nsym < 2u ? nsym : 2u;
            const uint32_t s2 = syms & (n2 == 2u ? 0xffffu : 0xffu);
            b.stab[x] = sm | (used << 16) | (nsym << 24);
            b.etab[x] = s2 | (used2 << 16) | (n2 << 24);
        }
        if (x < (1u << b.wf64)) {
            if (n4 == 0) {
                b.e64[2 * x] = 0;
                b.e64[2 * x + 1] = 0x3210u | (HB_E64_MARK << 26);
            } else {
                b.e64[2 * x] = n4 == 4u ? syms : (syms & ((1u << (8u * n4)) - 1u));
                b.e64[2 * x + 1] = (0x3210u + 0x1111u * n4) | ((8u * n4) << 16) | (used4 << 26);
            }
        }
        return;
    }
    const uint32_t k = i - nf;
    if (b.fsm && k < b.nstates * 256u) {
        const uint32_t s = k >> 8, byte = k & 255u;
        int32_t node = b.state_node[s];
        uint32_t ends = 0;
#pragma unroll
        for (int bit = 0; bit < 8; bit++) {
            node = ((byte >> bit) & 1u) ? b.tree[node].ione : b.tree[node].izero;
            if (b.tree[node].izero == -1) { ends++; node = 0; }
        }
        b.fsm[k] = (uint16_t)(((uint32_t)b.node_state[node] << 8) | ends);
    }
}

/* ------------------------------------------------------------------------- */
/* Sync kernel, fast path: FULL tiles of a code whose transducer fits shared memory
 * (hb_format.h; every byte-alphabet tree).  Same outputs as hb_sync_kernel -- the
 * (entry offset, starts) record of every subsequence and the tile's 32-entry map --
 * but the chains are followed by the byte-step transducer: 4 instructions per 8
 * stream bits (PRMT, LEA, LDS.U16, IADD), no data-dependent loop, no divergence.
 * A CTA holds ONE copy of the table (up to 128 KB) and G independent groups of
 * HB_T threads, each working on its own tile behind its own named barrier. */
#ifndef HB_FSM_CTAS1
#define HB_FSM_CTAS1 6      /* resident CTAs per SM the G = 1 / G = 2 variants are compiled for */
#endif
#ifndef HB_FSM_CTAS2
#define HB_FSM_CTAS2 3
#endif
struct hb_fsm_args {
    const uint16_t *tab;     /* nstates * 256 */
    const uint16_t *pstep;   /* 256 */
    const uint8_t *depth;    /* 256 */
    uint32_t nstates;
};

__device__ __forceinline__ void hb_group_sync(uint32_t id) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "n"(HB_T) : "memory");
}
__device__ __forceinline__ bool hb_group_or(uint32_t id, bool p) {
    uint32_t r;
    asm volatile("{\n\t.reg .pred q, r;\n\tsetp.ne.u32 q, %2, 0;\n\tbar.red.or.pred r, %1, %3, q;\n\t"
                 "selp.u32 %0, 1, 0, r;\n\t}"
                 : "=r"(r) : "r"(id), "r"((uint32_t)p), "n"(HB_T) : "memory");
    return r != 0u;
}

/* exclusive scan over the HB_T threads of a group; s_warp: >= 9 words of the group */
__device__ __forceinline__ uint32_t hb_group_exscan(uint32_t v, uint32_t *s_warp, uint32_t id,
                                                    uint32_t tg, uint32_t *total) {
    const uint32_t lane = tg & 31u, wid = tg >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += y;
    }
    if (lane == 31u) s_warp[wid] = inc;
    hb_group_sync(id);
    if (wid == 0u) {
        uint32_t x = (lane < HB_T / 32) ? s_warp[lane] : 0u;
        uint32_t xi = x;
#pragma unroll
        for (int d = 1; d < HB_T / 32; d <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, xi, d);
            if (lane >= (uint32_t)d) xi += y;
        }
        if (lane < HB_T / 32) s_warp[lane] = xi - x;
        if (lane == HB_T / 32 - 1) s_warp[HB_T / 32] = xi;
    }
    hb_group_sync(id);
    *total = s_warp[HB_T / 32];
    return s_warp[wid] + inc - v;
}

struct hb_global_words {
    const uint32_t *words;
    uint64_t base, nwords;
    __device__ __forceinline__ uint32_t operator()(uint32_t i) const {
        return base + i < nwords ? __ldg(words + base + i) : 0u;
    }
};

/* per-group shared memory of hb_fsm_sync_kernel, in 32-bit words */
template <int WPT>
__host__ __device__ constexpr uint32_t hb_fsm_group_words() {
    return (uint32_t)(WPT * HB_T / 2 + HB_T + HB_T + 16);
}

/* LC > 0: the table is held in 1 << LC copies on disjoint banks (hb_fsmc_* in hb_core.cuh): 2.1
 * instead of 3.05 wavefronts per lookup with four copies, for two more instructions per step. */
template <int WPT, int G, int LC>
__global__ void __launch_bounds__(G * HB_T, (G == 1 ? HB_FSM_CTAS1 : (G == 2 ? HB_FSM_CTAS2 : 1)))
hb_fsm_sync_kernel(hb_stream_args a, hb_fsm_args fa, uint32_t ntiles_full,
                   uint16_t *__restrict__ subs, uint32_t *__restrict__ tmaps) {
    constexpr int T = HB_T;
    extern __shared__ __align__(16) uint32_t smem[];
    constexpr uint32_t R = 1u << LC;
    uint16_t *s_tab = reinterpret_cast<uint16_t *>(smem);                  /* nstates * 256 entries, R copies */
    uint8_t *s_depth = reinterpret_cast<uint8_t *>(smem + fa.nstates * 128u * R);   /* 256 */
    uint16_t *s_pstep = reinterpret_cast<uint16_t *>(smem + fa.nstates * 128u * R + 64u);   /* 256 */
    const uint32_t g = threadIdx.x / T, t = threadIdx.x % T, bar = g + 1u;
    uint32_t *s_l1 = smem + fa.nstates * 128u * R + 192u;                  /* level 1 of the single-symbol table */
    uint32_t *s_grp = s_l1 + (1u << a.w1) + g * hb_fsm_group_words<WPT>();
    uint16_t *s_rec = reinterpret_cast<uint16_t *>(s_grp);                 /* WPT * T records */
    uint32_t *s_cs = s_grp + WPT * T / 2;                                  /* T: prefix of END counts */
    uint32_t *s_exit = s_cs + T;                                           /* T: state behind each subsequence */
    uint32_t *s_warp = s_exit + T;                                         /* 16; [12..15]: X0, exit depth */

    {   /* table: 16-byte copies by the whole CTA */
        if constexpr (LC == 0) {
            const uint4 *src = reinterpret_cast<const uint4 *>(fa.tab);
            uint4 *dst = reinterpret_cast<uint4 *>(s_tab);
            for (uint32_t i = threadIdx.x; i < fa.nstates * 32u; i += G * T) dst[i] = __ldg(src + i);
        } else {
            /* copy c of entry (s, b) at 16-bit index s * 256 R + (b >> lo) * 64 + c * (64 / R) + (b & mlo):
             * 4-byte pairs of entries stay together (lo >= 4) */
            constexpr uint32_t lo = 6u - LC, mlo = (1u << lo) - 1u;
            const uint32_t *src = reinterpret_cast<const uint32_t *>(fa.tab);
            uint32_t *dst = reinterpret_cast<uint32_t *>(s_tab);
            for (uint32_t i = threadIdx.x; i < fa.nstates * 128u; i += G * T) {
                const uint32_t v = __ldg(src + i), sb = 2u * i, st = sb >> 8, b = sb & 0xffu;
                const uint32_t at = st * 256u * R + (b >> lo) * 64u + (b & mlo);
#pragma unroll
                for (uint32_t c = 0; c < R; c++) dst[(at + c * (64u / R)) >> 1] = v;
            }
        }
        for (uint32_t i = threadIdx.x; i < 256u; i += G * T) {
            s_depth[i] = __ldg(fa.depth + i);
            s_pstep[i] = __ldg(fa.pstep + i);
        }
        /* three lanes in four turn their boundary state into a forward offset with one probe of this
         * table (hb_fsm_fwd): from global memory that was 20 tag lookups per warp and subsequence */
        for (uint32_t i = threadIdx.x; i < (1u << a.w1); i += G * T) s_l1[i] = __ldg(a.lut + i);
    }
    __syncthreads();
    hb_fsm f;
    f.tab = s_tab;
    f.tab_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_tab));
    f.depth = s_depth;
    f.pstep = s_pstep;
    f.lc = (uint32_t)LC;
    f.cbits = LC ? ((t & (R - 1u)) << (14 - 2 * LC)) * 0x10001u : 0u;
    const hb_lutref slow{s_l1, a.lut, (1u << a.w1) - 1u};

    /* w[WPT], the first word behind the subsequence, is only read by the tile's last thread */
    auto load_tile = [&](uint32_t tl, uint32_t (&w)[WPT + 1]) {
        const uint64_t wb = (uint64_t)tl * (T * WPT) + (uint64_t)t * WPT;
        hb_load_words<WPT, false>(a, wb, w);
        if (t == T - 1) w[WPT] = wb + WPT < a.nwords ? __ldg(a.words + wb + WPT) : 0u;
    };
    uint32_t tile = blockIdx.x * G + g;
    uint32_t w[WPT + 1];
    w[WPT] = 0u;
    if (tile < ntiles_full) load_tile(tile, w);
    while (tile < ntiles_full) {
        const uint64_t wbase = (uint64_t)tile * (T * WPT) + (uint64_t)t * WPT;

        /* chain of the guess "a codeword starts at bit 0 of my subsequence" */
        uint32_t rec[WPT];
        uint32_t st_in = 0u;
        uint32_t v[LC ? 2 * WPT : 2];          /* spread words (kept for the re-walks) */
        if constexpr (LC == 0) {
            hb_fsm_walk<WPT>(f, w, st_in, rec);
        } else {
#pragma unroll
            for (int j = 0; j < WPT; j++) hb_fsmc_spread<LC>(w[j], f.cbits, v[2 * j], v[2 * j + 1]);
            hb_fsmc_walk<WPT, LC>(f, v, st_in, rec);
        }
        s_exit[t] = hb_frec_state(rec[WPT - 1]);
        hb_group_sync(bar);

        /* stitch: my entering state is my left neighbour's exit state; repeat until no
         * exit state moves */
        for (;;) {
            bool changed = false;
            if (t > 0) {
                const uint32_t sn = s_exit[t - 1];
                if (sn != st_in) {
                    st_in = sn;
                    if constexpr (LC == 0) changed = hb_fsm_rewalk<WPT>(f, w, st_in, rec);
                    else changed = hb_fsmc_rewalk<WPT, LC>(f, v, st_in, rec);
                }
            }
            if (!hb_group_or(bar, changed)) break;
            s_exit[t] = hb_frec_state(rec[WPT - 1]);
            hb_group_sync(bar);
        }

        /* records in the pipeline's convention: forward entry offset, codeword STARTS */
        uint32_t ends = 0;
#pragma unroll
        for (int j = 0; j < WPT; j++) {
            ends += hb_frec_ends(rec[j]);
            s_rec[j * T + t] = (uint16_t)rec[j];
        }
        const uint32_t d_in = s_depth[st_in], d_out = s_depth[hb_frec_state(rec[WPT - 1])];
        uint32_t e = 0u;
        /* the word before my subsequence is my left neighbour's last one: a shuffle, and
         * one load per warp for lane 0 */
        uint32_t wprev = __shfl_up_sync(0xffffffffu, w[WPT - 1], 1);
        if ((t & 31u) == 0u && d_in) wprev = __ldg(a.words + wbase - 1);
        if (d_in) e = hb_fsm_fwd(slow, wprev, w[0], d_in);   /* t > 0 here */
        subs[(uint64_t)tile * T + t] = hb_sub_pack(e, ends - (d_in ? 1u : 0u) + (d_out ? 1u : 0u));
        if (t == T - 1) {
            s_warp[12] = hb_fsm_fwd(slow, w[WPT - 1], w[WPT], d_out);
            s_warp[13] = d_out;
        }
        /* the words are dead from here on: fetch the next tile's now, so that the loads
         * fly during the scan, the hypothesis walks and the barriers */
        const uint32_t next = tile + gridDim.x * G;
        if (next < ntiles_full) load_tile(next, w);
        uint32_t E0;
        s_cs[t] = hb_group_exscan(ends, s_warp, bar, t, &E0);
        hb_group_sync(bar);

        /* tile map: hypothesis 0 is the converged chain; 1..maxlen-1 are followed by
         * one lane each until they meet it */
        if (t < 32) {
            const uint32_t X0 = s_warp[12], d0 = s_warp[13];
            uint32_t m = hb_map_pack32(X0, E0 + (d0 ? 1u : 0u));
            if (t > 0 && t < a.maxlen && hb_entry_possible(a, tile, (uint32_t)(T * 32 * WPT), t)) {
                hb_global_words word{a.words, (uint64_t)tile * (T * WPT), a.nwords};
                m = hb_fsm_hyp_walk<WPT, T>(f, slow, word, s_rec, s_cs, E0, X0, d0, t);
            }
            tmaps[(uint64_t)tile * 32 + t] = m;
        }
        hb_group_sync(bar);
        tile = next;
    }
}

/* ------------------------------------------------------------------------- */
/* Map composition.  A warp holds 32 maps in registers (lane l = entry l) and
 * follows all 32 hypotheses at once with shuffles. */

__device__ __forceinline__ uint64_t hb_shfl64(uint64_t v, int src) {
    uint32_t lo = __shfl_sync(0xffffffffu, (uint32_t)v, src);
    uint32_t hi = __shfl_sync(0xffffffffu, (uint32_t)(v >> 32), src);
    return ((uint64_t)hi << 32) | lo;
}

/* up-sweep: per warp the composition of its 32 tile maps (wmaps), per CTA the
 * composition of its 32 warp maps (cmaps) */
__global__ void __launch_bounds__(HB_SCAN_T)
hb_scan_up_kernel(const uint32_t *__restrict__ tmaps, uint32_t ntiles,
                  uint64_t *__restrict__ wmaps, uint64_t *__restrict__ cmaps) {
    __shared__ uint64_t s_w[32][32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint64_t gw = (uint64_t)blockIdx.x * 32 + wid;
    uint32_t reg[32];
#pragma unroll
    for (int j = 0; j < 32; j++) {
        uint64_t tile = gw * 32 + j;
        reg[j] = tile < ntiles ? __ldg(tmaps + tile * 32 + lane) : hb_map_pack32(lane, 0);
    }
    uint32_t cur = lane, cnt = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        uint32_t m = __shfl_sync(0xffffffffu, reg[j], cur);
        cnt += m >> 8;
        cur = m & 31u;
    }
    uint64_t wm = hb_map_pack64(cur, cnt);
    wmaps[gw * 32 + lane] = wm;
    s_w[wid][lane] = wm;
    __syncthreads();
    if (wid == 0) {
        uint32_t c2 = lane;
        uint64_t n2 = 0;
#pragma unroll 4
        for (int j = 0; j < 32; j++) {
            uint64_t m = s_w[j][c2];
            n2 += m >> 8;
            c2 = (uint32_t)m & 31u;
        }
        cmaps[(uint64_t)blockIdx.x * 32 + lane] = hb_map_pack64(c2, n2);
    }
}

/* top: one warp walks the CTA maps in order; cprefix[c][e] = state of hypothesis
 * e on entering CTA c; shard_map[e] = state after the last CTA */
__global__ void __launch_bounds__(32)
hb_scan_top_kernel(const uint64_t *__restrict__ cmaps, uint32_t ncta,
                   uint64_t *__restrict__ cprefix, uint64_t *__restrict__ shard_map) {
    const int lane = threadIdx.x;
    uint32_t cur = lane;
    uint64_t cnt = 0;
    for (uint32_t c0 = 0; c0 < ncta; c0 += 32) {
        uint64_t reg[32];
#pragma unroll
        for (int j = 0; j < 32; j++)
            reg[j] = (c0 + j < ncta) ? __ldg(cmaps + (uint64_t)(c0 + j) * 32 + lane)
                                     : hb_map_pack64(lane, 0);
#pragma unroll
        for (int j = 0; j < 32; j++) {
            if (c0 + j < ncta) cprefix[(uint64_t)(c0 + j) * 32 + lane] = hb_map_pack64(cur, cnt);
            uint64_t m = hb_shfl64(reg[j], cur);
            cnt += m >> 8;
            cur = (uint32_t)m & 31u;
        }
    }
    shard_map[lane] = hb_map_pack64(cur, cnt);
}

/* rank composition after the all-gather: entry offset and output base of this
 * rank, total symbols of all ranks */
__global__ void hb_compose_kernel(const uint64_t *__restrict__ all_maps, int n_ranks,
                                  int rank, uint64_t *__restrict__ entry_base) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t cur = 0;
    uint64_t base = 0;
    for (int r = 0; r < n_ranks; r++) {
        if (r == rank) { entry_base[0] = cur; entry_base[1] = base; }
        uint64_t m = all_maps[(uint64_t)r * 32 + cur];
        base += m >> 8;
        cur = (uint32_t)m & 31u;
    }
    entry_base[2] = base;
}

/* One stream word of a tile for hb_fix_entries (0 past the end of the data). */
struct hb_tile_words {
    const uint32_t *words;
    uint64_t base, nwords;
    __device__ __forceinline__ uint32_t operator()(uint32_t i) const {
        return base + i < nwords ? __ldg(words + base + i) : 0u;
    }
};

/* down-sweep + fix: the entry offset and output base of every tile, and -- where a tile's
 * true entry offset differs from the hypothesis the sync kernel recorded (0) -- the
 * (entry, count) records of its leading subsequences (typically 1-2) re-chained in place
 * by the thread that owns the tile (S-table; fixed-length codes: hb_fix_fixed_kernel).
 * result[0] = symbols of this shard, [1] = exit offset, [2] = entry, [3] = base.
 * Launched after hb_scan_top_kernel. */
/* cmaps != nullptr ("no top" mode; single shard whose map nobody reads between the phases, at most
 * HB_NOTOP_MAX_CTAS scan CTAs): hb_scan_top_kernel was not launched -- CTA b stages the maps of the
 * CTAs before it in (dynamic) shared memory and one thread follows the ONE chain that matters, that
 * of the shard's entry offset, through them (b dependent shared-memory reads instead of a launch);
 * the last CTA goes on through its own map and writes the result. */
#define HB_NOTOP_MAX_CTAS 120
template <int WPT>
__global__ void __launch_bounds__(HB_SCAN_T)
hb_scan_downfix_kernel(hb_stream_args a, const uint32_t *__restrict__ tmaps,
                       const uint64_t *__restrict__ wmaps, const uint64_t *__restrict__ cprefix,
                       const uint64_t *__restrict__ shard_map,
                       const uint64_t *__restrict__ entry_base,
                       uint8_t *__restrict__ tile_entry, uint64_t *__restrict__ tile_base,
                       uint64_t *__restrict__ result, uint16_t *__restrict__ subs,
                       const uint64_t *__restrict__ cmaps) {
    constexpr int T = HB_T;
    constexpr uint32_t TS = T * 32u * WPT;
    __shared__ __align__(16) uint32_t s_fast[1u << HB_WF_MAX];   /* S-table, for the fix step */
    __shared__ uint32_t s_we[32];
    __shared__ uint64_t s_wb[32];
    __shared__ uint64_t s_cp;
    extern __shared__ __align__(16) uint64_t s_cm[];              /* "no top" mode: gridDim.x x 32 CTA maps */
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t ntiles = a.ntiles;
    const bool fixed_len = a.minlen == a.maxlen;
    if (!fixed_len)
        for (uint32_t i = threadIdx.x; i < (1u << a.wf); i += HB_SCAN_T) s_fast[i] = __ldg(a.fast + i);
    const uint32_t E = entry_base ? (uint32_t)entry_base[0] & 31u : 0u;
    const uint64_t B = entry_base ? entry_base[1] : 0ull;
    uint64_t cp;
    if (cmaps) {
        const bool last = blockIdx.x == gridDim.x - 1;
        const uint32_t nrows = blockIdx.x + (last ? 1u : 0u);
        for (uint32_t i = threadIdx.x; i < nrows * 32u; i += HB_SCAN_T) s_cm[i] = __ldg(cmaps + i);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t cur = E;
            uint64_t n = 0;
            for (uint32_t c = 0; c < blockIdx.x; c++) {
                const uint64_t m = s_cm[c * 32u + cur];
                n += m >> 8;
                cur = (uint32_t)m & 31u;
            }
            s_cp = hb_map_pack64(cur, n);
            if (last) {
                const uint64_t m = s_cm[blockIdx.x * 32u + cur];
                uint64_t total = n + (m >> 8);
                const uint32_t x = (uint32_t)m & 31u;
                if (total && a.bits_own + x > a.bits_avail) total--;   /* see below */
                result[0] = total;
                result[1] = x;
                result[2] = E;
                result[3] = B;
            }
        }
        __syncthreads();
        cp = s_cp;
    } else {
        cp = __ldg(cprefix + (uint64_t)blockIdx.x * 32 + E);
    }
    if (!cmaps && blockIdx.x == 0 && threadIdx.x == 0) {
        uint64_t sm = shard_map[E];
        uint64_t total = sm >> 8;
        /* the serial decoder emits a symbol only on reaching a leaf: a last
         * codeword that runs past the end of the data is not a symbol */
        if (total && a.bits_own + (sm & 31u) > a.bits_avail) total--;
        result[0] = total;
        result[1] = sm & 31u;
        result[2] = E;
        result[3] = B;
    }
    if (wid == 0) {
        uint64_t reg[32];
#pragma unroll
        for (int j = 0; j < 32; j++)
            reg[j] = __ldg(wmaps + ((uint64_t)blockIdx.x * 32 + j) * 32 + lane);
        uint32_t cur = (uint32_t)cp & 31u;
        uint64_t b = cp >> 8;      /* offsets are local to this shard's output buffer */
        uint32_t my_e = 0;
        uint64_t my_b = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            if (lane == j) { my_e = cur; my_b = b; }
            uint64_t m = hb_shfl64(reg[j], cur);
            b += m >> 8;
            cur = (uint32_t)m & 31u;
        }
        s_we[lane] = my_e;
        s_wb[lane] = my_b;
    }
    __syncthreads();
    const uint64_t gw = (uint64_t)blockIdx.x * 32 + wid;
    uint32_t reg[32];
#pragma unroll
    for (int j = 0; j < 32; j++) {
        uint64_t tile = gw * 32 + j;
        reg[j] = tile < ntiles ? __ldg(tmaps + tile * 32 + lane) : hb_map_pack32(lane, 0);
    }
    uint32_t cur = s_we[wid];
    uint64_t b = s_wb[wid];
    uint32_t my_e = 0;
    uint64_t my_b = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        if (lane == j) { my_e = cur; my_b = b; }
        uint32_t m = __shfl_sync(0xffffffffu, reg[j], cur);
        b += m >> 8;
        cur = m & 31u;
    }
    const uint64_t tile = gw * 32 + lane;
    if (tile >= ntiles) return;
    tile_entry[tile] = (uint8_t)my_e;
    tile_base[tile] = my_b;
    if (my_e == 0 || fixed_len) return;
    hb_tables tb;
    tb.fast = s_fast;
    tb.fast_saddr = (uint32_t)__cvta_generic_to_shared(s_fast);
    tb.fmask4 = ((1u << a.wf) - 1u) << 2;
    tb.slow = hb_lutref{a.lut, a.lut, (1u << a.w1) - 1u};
    const uint64_t own_left = a.bits_own - tile * TS;
    const uint32_t tile_lim = own_left < TS ? (uint32_t)own_left : TS;
    hb_tile_words word{a.words, tile * (T * WPT), a.nwords};
    hb_fix_entries<WPT, T>(tb, word, subs + tile * T, tile_lim, my_e);
}

/* ------------------------------------------------------------------------- */
/* Small streams (at most 1024 tiles = one scan CTA, single shard): hb_scan_up, _top,
 * _down and hb_fix in ONE launch.  The shipped corpora are a few hundred tiles; for
 * them four dependent tiny kernels cost more than the sync and emit kernels together
 * (tools/latency_probe.py).  Same results in the same buffers; the tile maps stay in
 * registers between the up and the down sweep. */
template <int WPT>
__global__ void __launch_bounds__(HB_SCAN_T)
hb_scan_small_kernel(hb_stream_args a, const uint32_t *__restrict__ tmaps,
                     const uint64_t *__restrict__ entry_base, uint64_t *__restrict__ shard_map,
                     uint8_t *__restrict__ tile_entry, uint64_t *__restrict__ tile_base,
                     uint64_t *__restrict__ result, uint16_t *__restrict__ subs) {
    constexpr int T = HB_T;
    constexpr uint32_t TS = T * 32u * WPT;
    __shared__ __align__(16) uint32_t s_fast[1u << HB_WF_MAX];   /* S-table, for the fix step */
    __shared__ uint64_t s_w[32][32];
    __shared__ uint32_t s_we[32];
    __shared__ uint64_t s_wb[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool fixed_len = a.minlen == a.maxlen;
    if (!fixed_len)
        for (uint32_t i = threadIdx.x; i < (1u << a.wf); i += HB_SCAN_T) s_fast[i] = __ldg(a.fast + i);

    /* up: the composition of this warp's 32 tile maps, all 32 hypotheses at once */
    uint32_t reg[32];
#pragma unroll
    for (int j = 0; j < 32; j++) {
        const uint32_t tile = (uint32_t)wid * 32u + j;
        reg[j] = tile < a.ntiles ? __ldg(tmaps + (uint64_t)tile * 32 + lane) : hb_map_pack32(lane, 0);
    }
    {
        uint32_t cur = lane, cnt = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            const uint32_t m = __shfl_sync(0xffffffffu, reg[j], cur);
            cnt += m >> 8;
            cur = m & 31u;
        }
        s_w[wid][lane] = hb_map_pack64(cur, cnt);
    }
    __syncthreads();
    if (wid == 0) {
        /* top: the shard's map (kept for hb_result); down over the warp maps from the
         * shard's entry offset */
        uint32_t c2 = lane;
        uint64_t n2 = 0;
#pragma unroll 4
        for (int j = 0; j < 32; j++) {
            const uint64_t m = s_w[j][c2];
            n2 += m >> 8;
            c2 = (uint32_t)m & 31u;
        }
        shard_map[lane] = hb_map_pack64(c2, n2);
        const uint32_t E = entry_base ? (uint32_t)entry_base[0] & 31u : 0u;
        const uint64_t B = entry_base ? entry_base[1] : 0ull;
        uint32_t cur = E;
        uint64_t b = 0;
#pragma unroll 4
        for (int j = 0; j < 32; j++) {
            if (lane == j) { s_we[j] = cur; s_wb[j] = b; }
            const uint64_t m = s_w[j][cur];
            b += m >> 8;
            cur = (uint32_t)m & 31u;
        }
        if (lane == 0) {
            /* a last codeword that runs past the end of the data is not a symbol */
            uint64_t total = b;
            if (total && a.bits_own + cur > a.bits_avail) total--;
            result[0] = total;
            result[1] = cur;
            result[2] = E;
            result[3] = B;
        }
    }
    __syncthreads();
    /* down inside the warp; lane j keeps tile j's entry offset and output base */
    uint32_t cur = s_we[wid], my_e = 0;
    uint64_t b = s_wb[wid], my_b = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        if (lane == j) { my_e = cur; my_b = b; }
        const uint32_t m = __shfl_sync(0xffffffffu, reg[j], cur);
        b += m >> 8;
        cur = m & 31u;
    }
    const uint32_t tile = (uint32_t)wid * 32u + lane;
    if (tile >= a.ntiles) return;
    tile_entry[tile] = (uint8_t)my_e;
    tile_base[tile] = my_b;
    /* fix: re-chain the head of a tile whose true entry offset is not the recorded 0
     * (fixed-length codes: hb_fix_fixed_kernel, launched by the host) */
    if (my_e == 0 || fixed_len) return;
    hb_tables tb;
    tb.fast = s_fast;
    tb.fast_saddr = (uint32_t)__cvta_generic_to_shared(s_fast);
    tb.fmask4 = ((1u << a.wf) - 1u) << 2;
    tb.slow = hb_lutref{a.lut, a.lut, (1u << a.w1) - 1u};
    const uint64_t own_left = a.bits_own - (uint64_t)tile * TS;
    const uint32_t tile_lim = own_left < TS ? (uint32_t)own_left : TS;
    hb_tile_words word{a.words, (uint64_t)tile * (T * WPT), a.nwords};
    hb_fix_entries<WPT, T>(tb, word, subs + (uint64_t)tile * T, tile_lim, my_e);
}

/* Fixed-length codes: the chain of the tile's true entry offset never meets the
 * recorded one, but every subsequence's (entry, count) follows arithmetically.
 * One thread per subsequence. */
template <int WPT>
__global__ void __launch_bounds__(HB_T)
hb_fix_fixed_kernel(hb_stream_args a, const uint8_t *__restrict__ tile_entry,
                    uint16_t *__restrict__ subs) {
    constexpr uint32_t S = 32u * WPT;
    constexpr uint32_t TS = HB_T * S;
    const uint32_t tile = blockIdx.x, t = threadIdx.x;
    const uint32_t E = tile_entry[tile];
    if (E == 0) return;
    const uint64_t own_left = a.bits_own - (uint64_t)tile * TS;
    const uint32_t tile_lim = own_left < TS ? (uint32_t)own_left : TS;
    const uint32_t s0 = t * S;
    if (s0 >= tile_lim) return;
    const uint32_t s1 = tile_lim - s0 < S ? tile_lim : s0 + S;
    const uint32_t first = hb_fixed_next(E, a.maxlen, s0);
    subs[(uint64_t)tile * HB_T + t] =
        hb_sub_pack((first - s0) & 31u, hb_fixed_count(E, a.maxlen, s0, s1));
}

/* ------------------------------------------------------------------------- */
/* Emit kernel, word-granular variant (hb_emit_words): staging stores of whole 32-bit
 * words assembled in a register window, each thread's last partial word stored
 * byte-wise after a barrier; software-pipelined tile loads; bulk-store wait deferred to
 * the next window.  Probes read the E64-table (up to four symbols per probe). */
#ifndef HB_EMITW_MIN_CTAS
#define HB_EMITW_MIN_CTAS 4
#endif
/* per-group shared memory in 32-bit words (16-byte multiple) */
__host__ __device__ __forceinline__ uint32_t hb_emitw_group_words(uint32_t stage_bytes) {
    return 16u + stage_bytes / 4u;
}

/* A CTA is G groups of HB_T threads, each on its own tile behind its own named barrier,
 * sharing ONE copy set of the E64-table (R = 1 << rshift copies, hb_tables64): with G = 2 and
 * R = 2 the table costs the same shared memory per thread as one copy per 256 threads, and
 * lanes 0-7 / 8-15 of each half-warp read different copies (different banks). */
template <int WPT, int G>
__global__ void __launch_bounds__(G * HB_T, HB_EMITW_MIN_CTAS / G)
hb_emitw_kernel(hb_stream_args a, uint32_t tile0, uint32_t rshift, const uint16_t *__restrict__ subs,
               const uint64_t *__restrict__ tile_base, const uint64_t *__restrict__ result, uint8_t *__restrict__ out,
               uint64_t out_capacity, uint32_t win, uint32_t stage_bytes, uint32_t *__restrict__ status) {
    constexpr int T = HB_T;
    constexpr uint32_t S = 32u * WPT;
    constexpr uint32_t TS = T * S;
    constexpr uint32_t EW = 2u;                            /* words per E64 entry */
    extern __shared__ __align__(16) uint32_t smem[];
    const uint32_t g = threadIdx.x / T, t = threadIdx.x % T, bar = g + 1u;
    uint32_t *s_fast = smem;                               /* E64-table: (2 << a.wf) << rshift words */
    uint32_t *s_warp = smem + ((EW << a.wf) << rshift) + g * hb_emitw_group_words(stage_bytes);   /* 16 */
    uint8_t *s_out = reinterpret_cast<uint8_t *>(s_warp + 16);   /* staging, 16-aligned */

    {
        const uint2 *src = reinterpret_cast<const uint2 *>(a.fast);
        uint2 *dst = reinterpret_cast<uint2 *>(s_fast);
        for (uint32_t i = threadIdx.x; i < ((1u << a.wf) << rshift); i += G * T) dst[i] = __ldg(src + (i >> rshift));
    }
    __syncthreads();
    hb_tables64 tb64;
    tb64.fast = s_fast;
    tb64.fast_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_fast));
    tb64.sc = 3u + rshift;
    tb64.fmask = ((1u << a.wf) - 1u) << tb64.sc;
    /* a half-warp (one LDS.64 wavefront group) spreads over all copies */
    tb64.laneoff = hb_opaque(((t >> (4u - rshift)) & ((1u << rshift) - 1u)) << 3);   /* rshift <= 4 */
    tb64.slow = hb_lutref{a.lut, a.lut, (1u << a.w1) - 1u};
    const uint64_t total_valid = result[0];
    const uint32_t s_out_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_out));

    /* software pipeline: the next tile's words, record and output base are fetched as
     * soon as this tile's words are dead (after its last decode window), so that the
     * loads fly during the copy-out, the barriers and the next scan */
    const uint32_t tstep = gridDim.x * G;
    uint32_t tile = tile0 + blockIdx.x * G + g, nwin = 0;
    uint32_t w[WPT + 1];
    uint16_t sub = 0;
    uint64_t B = 0;
    if (tile < a.ntiles) {
        hb_load_words<WPT>(a, (uint64_t)tile * (T * WPT) + (uint64_t)t * WPT, w);
        sub = subs[(uint64_t)tile * T + t];   /* already re-chained by the down-sweep kernel */
        B = tile_base[tile];
    }
    while (tile < a.ntiles) {
        const uint64_t tile_bit0 = (uint64_t)tile * TS;
        const uint64_t sub0 = tile_bit0 + (uint64_t)t * S;
        const uint32_t next = tile + tstep;
        const uint64_t Bt = B;

        const uint32_t e = hb_sub_entry(sub), c = hb_sub_count(sub);
        uint32_t nk;
        const uint32_t o = hb_group_exscan(c, s_warp, bar, t, &nk);
        const uint32_t lim = sub0 >= a.bits_own ? 0u
                           : (a.bits_own - sub0 < S ? (uint32_t)(a.bits_own - sub0) : S);
        /* symbols past the shard's valid total (a cut-off last codeword) are not written */
        uint32_t nvalid = nk;
        if (Bt >= total_valid) nvalid = 0;
        else if (Bt + nk > total_valid) nvalid = (uint32_t)(total_valid - Bt);
        const bool full_out = Bt + nvalid > out_capacity;
        if (full_out && t == 0) atomicOr(status, HB_ST_OUTPUT_FULL);

        /* The staging buffer holds `win` bytes of tile output plus one thread's
         * worth of overhang; a tile whose output is larger (data far more
         * compressible than the code table suggests) is emitted in several
         * windows.  Window p takes the threads whose first byte lies in
         * [p*win, (p+1)*win); their slices are contiguous, so it copies out
         * [end of window p-1's threads, end of its own threads). */
        uint32_t lo_b = 0;
        for (uint32_t wb = 0; !full_out && (wb == 0 || wb < nk); wb += win, nwin++) {
            const bool mine = c && o >= wb && o - wb < win;
            const bool last_win = wb + win >= nk;
            const uint32_t al = (uint32_t)((reinterpret_cast<uintptr_t>(out) + Bt + wb) & 15u);
            uint32_t *s_hi = s_warp + 14 + (nwin & 1u);     /* alternating slot: no barrier after the copy-out */
            if (t == 0) {
                /* the previous window's bulk store must have read the staging buffer */
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                *s_hi = nk;                                  /* default: last window */
            }
            hb_group_sync(bar);
            hb_tail tl;
            tl.k = 0u;
            if (mine) {
                const hb_out_t dst = (hb_out_t)(s_out_saddr + al + (o - wb));
                if (lim != S) hb_emit_clipped<WPT>(tb64, w, lim, e, c, dst);
                else tl = hb_emit_words<WPT>(tb64, w, e, c, dst, (uint32_t)(uintptr_t)dst & 3u);
                if (o + c - wb >= win && o + c < nk) *s_hi = o + c;   /* I am the window's last thread */
            }
            if (last_win && next < a.ntiles) {
                hb_load_words<WPT>(a, (uint64_t)next * (T * WPT) + (uint64_t)t * WPT, w);
                sub = subs[(uint64_t)next * T + t];
                B = tile_base[next];
            }
            hb_group_sync(bar);
            /* every word store is done: the last, partial word of each slice (its other
             * lanes belong to the right neighbour, who has just overwritten them) */
            hb_store_tail(tl);
            /* every thread orders its own staging writes before the async proxy (the bulk
             * store below reads them), then the barrier orders the threads */
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            hb_group_sync(bar);
            uint32_t hi_b = *s_hi;
            if (hi_b > nvalid) hi_b = nvalid;
            if (lo_b < hi_b) {
                /* staging -> global: s_out[al + (b - wb)] -> out[B + b].  The staging index
                 * is congruent to the global address mod 16, so the 16-byte-aligned middle
                 * goes out as ONE bulk asynchronous copy (TMA, cp.async.bulk) issued by a
                 * single thread; the partial first / last vectors are stored byte-wise. */
                uint8_t *gbase = out + Bt + wb - al;          /* 16-byte aligned */
                const uint32_t begb = al + (lo_b - wb), endb = al + (hi_b - wb);
                const uint32_t a0 = (begb + 15u) & ~15u, a1 = endb & ~15u;
                if (a0 < a1) {
                    if (t == 0) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     :: "l"(gbase + a0), "r"(s_out_saddr + a0), "r"(a1 - a0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    if (t >= 32 && t < 64) {                 /* head and tail bytes, one warp */
                        const uint32_t i = t - 32;
                        if (begb + i < a0) gbase[begb + i] = s_out[begb + i];
                        if (a1 + i < endb) gbase[a1 + i] = s_out[a1 + i];
                    }
                } else {
                    for (uint32_t i = begb + t; i < endb; i += T) gbase[i] = s_out[i];   /* < 32 bytes */
                }
            }
            lo_b = hi_b > lo_b ? hi_b : lo_b;
        }
        if (full_out && next < a.ntiles) {
            hb_load_words<WPT>(a, (uint64_t)next * (T * WPT) + (uint64_t)t * WPT, w);
            sub = subs[(uint64_t)next * T + t];
            B = tile_base[next];
            hb_group_sync(bar);      /* the scan of the next tile reuses s_warp */
        }
        tile = next;
    }
    /* the staging buffer must outlive the last bulk store's reads */
    if (t == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

/* ------------------------------------------------------------------------- */
/* Emit kernel with 32-bit table entries (hb_emit_words32 in hb_core.cuh): the default for large
 * streams.  Same tile pipeline as hb_emitw_kernel; the differences are the table and the probe
 * loops.
 *   - The E32-table (a.fast, a.wf index bits; built once per codebook by hb_build_e32_kernel) is copied
 *     into shared memory in R = 1 << rshift copies interleaved entry by entry: copy r on banks r,
 *     r + R, ...; lane l reads copy l & (R - 1), so that only the 32 / R lanes of one copy can collide.
 *   - The table sits at a shared-memory address that is a multiple of its size (tab_off, computed
 *     by the host from the dynamic window's base address), so that "base | index | copy" is ONE
 *     LOP3 and the probe's address needs no add.  The groups' staging buffers fill the room in
 *     front of the table first (n_before of them), the rest follow it. */
#define HB_ST_LAYOUT 2u       /* the E32-table is not aligned to its size: host / device layout mismatch */
/* ADD: a table too large to be aligned to its size (15 index bits, 128 KB): at offset 0, one add per probe */
template <int WPT, int G, bool ADD>
__global__ void __launch_bounds__(G * HB_T, HB_EMITW_MIN_CTAS / G)
hb_emit32_kernel(hb_stream_args a, uint32_t tile0, uint32_t rshift, uint32_t tab_off, uint32_t n_before,
                 const uint16_t *__restrict__ subs, const uint64_t *__restrict__ tile_base,
                 const uint64_t *__restrict__ result, uint8_t *__restrict__ out, uint64_t out_capacity,
                 uint32_t win, uint32_t stage_bytes, uint32_t *__restrict__ status) {
    constexpr int T = HB_T;
    constexpr uint32_t S = 32u * WPT;
    constexpr uint32_t TS = T * S;
    extern __shared__ __align__(16) uint32_t smem[];
    const uint32_t g = threadIdx.x / T, t = threadIdx.x % T, bar = g + 1u;
    const uint32_t tab_bytes = 4u << (a.wf + rshift);
    const uint32_t grp = hb_emitw_group_words(stage_bytes);
    uint32_t *s_fast = smem + tab_off / 4u;
    uint32_t *s_warp = smem + (g < n_before ? g * grp : (tab_off + tab_bytes) / 4u + (g - n_before) * grp);   /* 16 */
    uint8_t *s_out = reinterpret_cast<uint8_t *>(s_warp + 16);   /* staging, 16-aligned */
    const uint32_t tab_saddr = (uint32_t)__cvta_generic_to_shared(s_fast);
    if (!ADD && (tab_saddr & (tab_bytes - 1u))) {
        if (threadIdx.x == 0) atomicOr(status, HB_ST_LAYOUT);
        return;
    }
    const hb_lutref slow{a.lut, a.lut, (1u << a.w1) - 1u};
    if (rshift == 0u) {       /* one copy: 16-byte vectors */
        const uint4 *src = reinterpret_cast<const uint4 *>(a.fast);
        uint4 *dst = reinterpret_cast<uint4 *>(s_fast);
        for (uint32_t i = threadIdx.x; i < (1u << a.wf) / 4u; i += G * T) dst[i] = __ldg(src + i);
    } else {
        for (uint32_t x = threadIdx.x; x < (1u << a.wf); x += G * T) {
            const uint32_t ent = __ldg(a.fast + x);
            for (uint32_t r = 0; r < (1u << rshift); r++) s_fast[(x << rshift) + r] = ent;
        }
    }
    __syncthreads();
    hb_tables32 tb;
    tb.fast = s_fast;
    tb.sc = 2u + rshift;
    tb.wf = a.wf;
    tb.fmask = ((1u << a.wf) - 1u) << tb.sc;
    tb.lanebase = hb_opaque((ADD ? 0u : tab_saddr) | ((t & ((1u << rshift) - 1u)) << 2));
    tb.addbase = hb_opaque(tab_saddr);
    tb.slow = slow;
    const uint64_t total_valid = result[0];
    const uint32_t s_out_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_out));

    const uint32_t tstep = gridDim.x * G;
    uint32_t tile = tile0 + blockIdx.x * G + g, nwin = 0;
    uint32_t w[WPT + 1];
    uint16_t sub = 0;
    uint64_t B = 0;
    if (tile < a.ntiles) {
        hb_load_words<WPT>(a, (uint64_t)tile * (T * WPT) + (uint64_t)t * WPT, w);
        sub = subs[(uint64_t)tile * T + t];
        B = tile_base[tile];
    }
    while (tile < a.ntiles) {
        const uint64_t tile_bit0 = (uint64_t)tile * TS;
        const uint64_t sub0 = tile_bit0 + (uint64_t)t * S;
        const uint32_t next = tile + tstep;
        const uint64_t Bt = B;

        const uint32_t e = hb_sub_entry(sub), c = hb_sub_count(sub);
        uint32_t nk;
        const uint32_t o = hb_group_exscan(c, s_warp, bar, t, &nk);
        const uint32_t lim = sub0 >= a.bits_own ? 0u
                           : (a.bits_own - sub0 < S ? (uint32_t)(a.bits_own - sub0) : S);
        uint32_t nvalid = nk;
        if (Bt >= total_valid) nvalid = 0;
        else if (Bt + nk > total_valid) nvalid = (uint32_t)(total_valid - Bt);
        const bool full_out = Bt + nvalid > out_capacity;
        if (full_out && t == 0) atomicOr(status, HB_ST_OUTPUT_FULL);

        /* windows: see hb_emitw_kernel */
        uint32_t lo_b = 0;
        for (uint32_t wb = 0; !full_out && (wb == 0 || wb < nk); wb += win, nwin++) {
            const bool mine = c && o >= wb && o - wb < win;
            const bool last_win = wb + win >= nk;
            const uint32_t al = (uint32_t)((reinterpret_cast<uintptr_t>(out) + Bt + wb) & 15u);
            uint32_t *s_hi = s_warp + 14 + (nwin & 1u);
            if (t == 0) {
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                *s_hi = nk;
            }
            hb_group_sync(bar);
            hb_tail tl;
            tl.k = 0u;
            if (mine) {
                const hb_out_t dst = (hb_out_t)(s_out_saddr + al + (o - wb));
                if (lim != S) hb_emit_clipped32<WPT, ADD>(tb, w, lim, e, c, dst);
                else tl = hb_emit_words32<WPT, ADD>(tb, w, e, c, dst, (uint32_t)(uintptr_t)dst & 3u);
                if (o + c - wb >= win && o + c < nk) *s_hi = o + c;
            }
            if (last_win && next < a.ntiles) {
                hb_load_words<WPT>(a, (uint64_t)next * (T * WPT) + (uint64_t)t * WPT, w);
                sub = subs[(uint64_t)next * T + t];
                B = tile_base[next];
            }
            hb_group_sync(bar);
            hb_store_tail(tl);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            hb_group_sync(bar);
            uint32_t hi_b = *s_hi;
            if (hi_b > nvalid) hi_b = nvalid;
            if (lo_b < hi_b) {
                uint8_t *gbase = out + Bt + wb - al;          /* 16-byte aligned */
                const uint32_t begb = al + (lo_b - wb), endb = al + (hi_b - wb);
                const uint32_t a0 = (begb + 15u) & ~15u, a1 = endb & ~15u;
                if (a0 < a1) {
                    if (t == 0) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     :: "l"(gbase + a0), "r"(s_out_saddr + a0), "r"(a1 - a0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    if (t >= 32 && t < 64) {
                        const uint32_t i = t - 32;
                        if (begb + i < a0) gbase[begb + i] = s_out[begb + i];
                        if (a1 + i < endb) gbase[a1 + i] = s_out[a1 + i];
                    }
                } else {
                    for (uint32_t i = begb + t; i < endb; i += T) gbase[i] = s_out[i];
                }
            }
            lo_b = hi_b > lo_b ? hi_b : lo_b;
        }
        if (full_out && next < a.ntiles) {
            hb_load_words<WPT>(a, (uint64_t)next * (T * WPT) + (uint64_t)t * WPT, w);
            sub = subs[(uint64_t)next * T + t];
            B = tile_base[next];
            hb_group_sync(bar);
        }
        tile = next;
    }
    if (t == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

/* ------------------------------------------------------------------------- */
/* Warp-autonomous emit kernel (E32-table): every WARP works through the stream on its own -- 32
 * consecutive subsequences (a "warp tile", an eighth of a sync tile) at a time, with its own staging
 * slice and its own TMA bulk store, ordered by __syncwarp only.  hb_emit32_kernel's groups of 256
 * threads meet at five named barriers per tile and wait there for their slowest warp (13 % of the
 * warps' time); here nothing waits for another warp.
 *   output base of a warp tile = the sync tile's base (down-sweep) + the symbols of the tile's
 *   subsequences in front of it: every lane sums 8 of the tile's 256 records (one 16-byte load),
 *   a warp scan of those sums gives the prefix at every 8th subsequence, lane 4 q holds warp tile q's.
 *   The staging slice holds `win` bytes plus one thread's overhang; a warp tile with more output
 *   goes out in several windows, exactly as in the group kernels. */
/* SPL = 2: a lane takes TWO consecutive subsequences (a warp tile is 64 of them, a quarter of a sync tile):
 * their output is contiguous and the chain runs on from one into the other (hb_emit_words32_part), so the
 * per-warp-tile prologue and epilogue -- 40 % of the kernel's instructions with SPL = 1 -- are paid once per
 * 512 stream bits instead of once per 256.  The second subsequence's words are loaded when the first is done.
 * Byte-exact, but measured slower than SPL = 1 (english1g 0.628 against 0.558 ms): an A/B path. */
/* E64 = true: the same warp-autonomous pipeline over the E64-table (up to FOUR symbols per probe, LDS.64; a.wf
 * index bits, 1 << rshift copies interleaved entry by entry as in hb_emitw_kernel) -- for codes so short that
 * three symbols do not fill a probe (the Fibonacci-skewed model: 2.6 bits per symbol).  SPL = 1 only. */
template <int WPT, bool ADD, int SPL, bool E64 = false>
__global__ void __launch_bounds__(1024, 1)
hb_emit32w_kernel(hb_stream_args a, uint32_t rshift, uint32_t tab_off, uint32_t stage_off,
                  const uint16_t *__restrict__ subs, const uint64_t *__restrict__ tile_base,
                  const uint64_t *__restrict__ result, uint8_t *__restrict__ out, uint64_t out_capacity,
                  uint32_t win, uint32_t stage_bytes, uint32_t *__restrict__ status) {
    constexpr int T = HB_T;
    constexpr uint32_t S = 32u * WPT;
    constexpr uint32_t UNIT = 32u * SPL;                    /* subsequences per warp tile */
    constexpr uint32_t WT = T / UNIT;                       /* warp tiles per sync tile */
    extern __shared__ __align__(16) uint32_t smem[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t tab_bytes = (E64 ? 8u : 4u) << (a.wf + rshift);
    uint32_t *s_fast = smem + tab_off / 4u;
    uint8_t *s_out = reinterpret_cast<uint8_t *>(smem) + stage_off + warp * stage_bytes;   /* 16-aligned */
    const uint32_t tab_saddr = (uint32_t)__cvta_generic_to_shared(s_fast);
    if (!E64 && !ADD && (tab_saddr & (tab_bytes - 1u))) {
        if (threadIdx.x == 0) atomicOr(status, HB_ST_LAYOUT);
        return;
    }
    if (E64) {
        const uint2 *src = reinterpret_cast<const uint2 *>(a.fast);
        uint2 *dst = reinterpret_cast<uint2 *>(s_fast);
        for (uint32_t i = threadIdx.x; i < ((1u << a.wf) << rshift); i += 1024u) dst[i] = __ldg(src + (i >> rshift));
    } else if (rshift == 0u) {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.fast);
        uint4 *dst = reinterpret_cast<uint4 *>(s_fast);
        for (uint32_t i = threadIdx.x; i < (1u << a.wf) / 4u; i += 1024u) dst[i] = __ldg(src + i);
    } else {
        for (uint32_t x = threadIdx.x; x < (1u << a.wf); x += 1024u) {
            const uint32_t ent = __ldg(a.fast + x);
            for (uint32_t r = 0; r < (1u << rshift); r++) s_fast[(x << rshift) + r] = ent;
        }
    }
    __syncthreads();
    hb_tables32 tb;
    tb.fast = s_fast;
    tb.sc = 2u + rshift;
    tb.wf = a.wf;
    tb.fmask = ((1u << a.wf) - 1u) << tb.sc;
    tb.lanebase = hb_opaque((ADD ? 0u : tab_saddr) | ((lane & ((1u << rshift) - 1u)) << 2));
    tb.addbase = hb_opaque(tab_saddr);
    tb.slow = hb_lutref{a.lut, a.lut, (1u << a.w1) - 1u};
    hb_tables64 tb64;
    tb64.fast = s_fast;
    tb64.fast_saddr = hb_opaque(tab_saddr);
    tb64.sc = 3u + rshift;
    tb64.fmask = ((1u << a.wf) - 1u) << tb64.sc;
    tb64.laneoff = hb_opaque(((lane >> (4u - rshift)) & ((1u << rshift) - 1u)) << 3);   /* rshift <= 4 */
    tb64.slow = tb.slow;
    const uint64_t total_valid = result[0];
    const uint32_t s_out_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_out));

    /* Warp `warp` of CTA b takes the units b * 32 + warp + k * (32 * gridDim.x): always the same eighth q of
     * a sync tile (32 * gridDim.x is a multiple of 8), so every address it needs advances by a constant. */
    const uint32_t nunits = a.ntiles * WT, ustep = gridDim.x * 32u;
    uint32_t u = blockIdx.x * 32u + warp;
    const uint32_t q = u % WT;
    const uint32_t *p_words = a.words + ((uint64_t)u * UNIT + lane * SPL) * WPT;
    const uint16_t *p_sub = subs + (uint64_t)u * UNIT + lane * SPL;
    const uint4 *p_rec8 = reinterpret_cast<const uint4 *>(subs + (uint64_t)(u / WT) * T) + lane;
    const uint64_t *p_base = tile_base + u / WT;
    const uint32_t *const words_end = a.words + a.nwords;
    const bool vec256 = (reinterpret_cast<uintptr_t>(a.words) & 31u) == 0;
    const bool cap_ok = total_valid <= out_capacity;        /* then no unit can overrun the output */
    uint32_t w[WPT + 1];
    uint32_t sub = 0;                                       /* my record(s): the second one in the high half */
    uint4 rec8 = make_uint4(0u, 0u, 0u, 0u);
    uint64_t B = 0;
    auto load_words = [&](const uint32_t *p_words) {
        if (p_words + WPT + 1 <= words_end) {
            if (WPT % 8 == 0 && vec256) {
#pragma unroll
                for (int v = 0; v < WPT / 8; v++)
                    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                                 : "=r"(w[8 * v]), "=r"(w[8 * v + 1]), "=r"(w[8 * v + 2]), "=r"(w[8 * v + 3]),
                                   "=r"(w[8 * v + 4]), "=r"(w[8 * v + 5]), "=r"(w[8 * v + 6]), "=r"(w[8 * v + 7])
                                 : "l"(p_words + 8 * v));
            } else {
#pragma unroll
                for (int v = 0; v < WPT / 4; v++) {
                    const uint4 x = __ldg(reinterpret_cast<const uint4 *>(p_words) + v);
                    w[4 * v + 0] = x.x; w[4 * v + 1] = x.y; w[4 * v + 2] = x.z; w[4 * v + 3] = x.w;
                }
            }
            /* SPL = 1: the word behind my subsequence is my right neighbour's first one -- a shuffle at the
             * top of the unit loop (one wavefront instead of nine tag lookups); only lane 31 loads it */
            if (SPL != 1 || lane == 31u) w[WPT] = __ldg(p_words + WPT);
        } else {
#pragma unroll
            for (int j = 0; j <= WPT; j++) w[j] = p_words + j < words_end ? __ldg(p_words + j) : 0u;
        }
    };
    auto fetch = [&]() {
        load_words(p_words);
        sub = SPL == 2 ? *reinterpret_cast<const uint32_t *>(p_sub) : (uint32_t)*p_sub;
        rec8 = __ldg(p_rec8);
        B = *p_base;
    };
    auto advance = [&]() {
        u += ustep;
        p_words += (uint64_t)ustep * UNIT * WPT;
        p_sub += (uint64_t)ustep * UNIT;
        p_rec8 += (uint64_t)(ustep / WT) * (T / 8);
        p_base += ustep / WT;
    };
    if (u < nunits) fetch();
    while (u < nunits) {
        if (SPL == 1) {
            const uint32_t nx = __shfl_down_sync(0xffffffffu, w[0], 1);
            if (lane != 31u) w[WPT] = nx;
        }
        const uint32_t e = hb_sub_entry((uint16_t)sub), c0 = hb_sub_count((uint16_t)sub);
        const uint32_t c = c0 + (SPL == 2 ? sub >> 21 : 0u);
        /* symbols of the sync tile's subsequences in front of this warp tile: the sum over the lanes below
         * 4 q of their 8 records (REDUX), the offset inside the warp tile by a scan */
        uint32_t s8 = (rec8.x & 0xffffu) >> 5;
        s8 += rec8.x >> 21;
        s8 += (rec8.y & 0xffffu) >> 5;
        s8 += rec8.y >> 21;
        s8 += (rec8.z & 0xffffu) >> 5;
        s8 += rec8.z >> 21;
        s8 += (rec8.w & 0xffffu) >> 5;
        s8 += rec8.w >> 21;
        const uint32_t front = __reduce_add_sync(0xffffffffu, lane < (UNIT / 8u) * q ? s8 : 0u);
        const uint32_t nk = __reduce_add_sync(0xffffffffu, c);
        uint32_t inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= (uint32_t)d) inc += y;
        }
        const uint32_t o = inc - c;
        const uint64_t Bt = B + front;
        if constexpr (!E64 && SPL == 1) {
            /* The common case, compiled on its own: the warp tile's output fits one window, and it is not in
             * the shard's last sync tile, so every subsequence is whole and every symbol valid.  The chains
             * end unclipped (hb_emit_words32_run); the window is [al, al + nk) of the slice. */
            if (nk <= win && u + WT < nunits && cap_ok) {
                const uint32_t al = (uint32_t)((reinterpret_cast<uintptr_t>(out) + Bt) & 15u);
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncwarp();
                const hb_out_t dst = (hb_out_t)(s_out_saddr + al + o);
                const hb_tail tl = hb_emit_words32_run<WPT, ADD>(tb, w, e, c, dst, (uint32_t)(uintptr_t)dst & 3u);
                advance();
                if (u < nunits) fetch();
                __syncwarp();                    /* every right neighbour's first store is done */
                hb_store_tail(tl);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                uint8_t *gbase = out + Bt - al;  /* 16-byte aligned */
                const uint32_t endb = al + nk, a0 = (al + 15u) & ~15u, a1 = endb & ~15u;
                if (a0 < a1) {
                    if (lane == 0) {
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     :: "l"(gbase + a0), "r"(s_out_saddr + a0), "r"(a1 - a0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    /* fewer than 16 bytes each: the head on lanes 0-15, the tail on lanes 16-31 */
                    const uint32_t i = lane < 16u ? al + lane : a1 + (lane - 16u);
                    if (i < (lane < 16u ? a0 : endb)) gbase[i] = s_out[i];
                } else if (al + lane < endb) {
                    gbase[al + lane] = s_out[al + lane];   /* < 32 bytes */
                }
                continue;
            }
        }
        /* Only in the shard's last sync tile can the stream end inside a subsequence, or the shard's last
         * codeword be cut off (its symbol is then not part of total_valid): everywhere else every
         * subsequence is whole and every symbol valid, and the 64-bit bookkeeping is skipped. */
        uint32_t lim = SPL * S, nvalid = nk;                /* owned bits of my SPL subsequences */
        bool full_out = false;
        if (u + WT >= nunits || !cap_ok) {
            const uint64_t sub0 = ((uint64_t)u * UNIT + lane * SPL) * S;
            lim = sub0 >= a.bits_own ? 0u : (a.bits_own - sub0 < SPL * S ? (uint32_t)(a.bits_own - sub0) : SPL * S);
            if (Bt >= total_valid) nvalid = 0;
            else if (total_valid - Bt < nk) nvalid = (uint32_t)(total_valid - Bt);
            full_out = Bt + nvalid > out_capacity;
            if (full_out && lane == 0) atomicOr(status, HB_ST_OUTPUT_FULL);
        }
        const uint32_t unext = u + ustep;

        uint32_t lo_b = 0;
        for (uint32_t wb = 0; !full_out && (wb == 0 || wb < nk); wb += win) {
            const bool mine = c && o >= wb && o - wb < win;
            const bool last_win = wb + win >= nk;
            const uint32_t al = (uint32_t)((reinterpret_cast<uintptr_t>(out) + Bt + wb) & 15u);
            /* the previous bulk store must have read the staging slice */
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            __syncwarp();
            hb_tail tl;
            tl.k = 0u;
            if (mine) {
                const hb_out_t dst = (hb_out_t)(s_out_saddr + al + (o - wb));
                if constexpr (E64) {
                    if (lim != S) hb_emit_clipped<WPT>(tb64, w, lim, e, c, dst);
                    else tl = hb_emit_words<WPT>(tb64, w, e, c, dst, (uint32_t)(uintptr_t)dst & 3u);
                } else if (lim != SPL * S) {
                    /* the stream ends inside this lane's bits: every subsequence on its own, byte stores */
                    hb_emit_clipped32<WPT, ADD>(tb, w, lim < S ? lim : S, e, c0, dst);
                    if (SPL == 2) {
                        load_words(p_words + WPT);
                        hb_emit_clipped32<WPT, ADD>(tb, w, lim > S ? lim - S : 0u, (sub >> 16) & 31u, c - c0, dst + c0);
                    }
                } else {
                    hb_w32 st;
                    hb_w32_begin(st, e, dst, (uint32_t)(uintptr_t)dst & 3u);
#pragma unroll 1
                    for (int h = 0; h < SPL; h++) {
                        if (h) load_words(p_words + WPT);
                        hb_emit_words32_part<WPT, ADD>(tb, w, st, c, dst, h == SPL - 1);
                    }
                    tl = hb_w32_tail(st);
                }
            }
            /* the window ends behind its last thread's slice (or with the warp tile) */
            const uint32_t cross = __ballot_sync(0xffffffffu, mine && o + c - wb >= win && o + c < nk);
            uint32_t hi_b = __shfl_sync(0xffffffffu, o + c, cross ? (int)hb_ctz(cross) : 0);
            if (!cross) hi_b = nk;
            if (last_win && unext < nunits) { advance(); fetch(); }
            __syncwarp();
            hb_store_tail(tl);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (hi_b > nvalid) hi_b = nvalid;
            if (lo_b < hi_b) {
                uint8_t *gbase = out + Bt + wb - al;          /* 16-byte aligned */
                const uint32_t begb = al + (lo_b - wb), endb = al + (hi_b - wb);
                const uint32_t a0 = (begb + 15u) & ~15u, a1 = endb & ~15u;
                if (a0 < a1) {
                    if (lane == 0) {
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     :: "l"(gbase + a0), "r"(s_out_saddr + a0), "r"(a1 - a0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    if (begb + lane < a0) gbase[begb + lane] = s_out[begb + lane];
                    if (a1 + lane < endb) gbase[a1 + lane] = s_out[a1 + lane];
                } else {
                    if (begb + lane < endb) gbase[begb + lane] = s_out[begb + lane];   /* < 32 bytes */
                }
            }
            lo_b = hi_b > lo_b ? hi_b : lo_b;
        }
        if (u != unext) {                        /* not advanced inside the window loop */
            advance();
            if (u < nunits) fetch();
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

/* ------------------------------------------------------------------------- */
/* Emit kernel, flat variant (hb_emit_flat in hb_core.cuh): full tiles that are not the last
 * tile of the shard.  A CTA is G groups of HB_T threads, each on its own tile behind its own
 * named barrier, sharing ONE EP-table built in shared memory by the CTA itself (R copies,
 * hb_format.h).  Per tile: the words go to shared memory transposed (word j of thread t at
 * [j][t]: a thread's reads stay in its own bank whatever j is), rows WPT.. hold the first
 * words of the next subsequence (the chain runs on into it until its last staging word is
 * complete); group scan of the counts; the decode; barrier; every thread stores its final
 * word once more (its right neighbour's first store has zeros in the shared lanes); the
 * 16-byte-aligned middle of the window leaves as one TMA bulk copy. */
#define HB_EMITF_LA 6       /* look-ahead rows: the chain may run (4 * 32 + 31 + 24) bits past the subsequence */
template <int WPT>
__host__ __device__ constexpr uint32_t hb_emitf_group_words(uint32_t stage_bytes) {
    return 16u + (uint32_t)(WPT + HB_EMITF_LA) * HB_T + stage_bytes / 4u;
}

struct hb_col_smem {        /* a thread's column of the transposed tile */
    uint32_t p, stride;
    __device__ __forceinline__ uint32_t next() {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(p));
        p += stride;
        return v;
    }
};

template <int WPT>
__device__ __forceinline__ void hb_load_words_n(const hb_stream_args &a, uint64_t wbase, uint32_t (&w)[WPT]) {
    if (wbase + WPT <= a.nwords) {
        if (WPT % 8 == 0 && (reinterpret_cast<uintptr_t>(a.words) & 31u) == 0) {
#pragma unroll
            for (int v = 0; v < WPT / 8; v++)
                asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                             : "=r"(w[8 * v]), "=r"(w[8 * v + 1]), "=r"(w[8 * v + 2]), "=r"(w[8 * v + 3]),
                               "=r"(w[8 * v + 4]), "=r"(w[8 * v + 5]), "=r"(w[8 * v + 6]), "=r"(w[8 * v + 7])
                             : "l"(a.words + wbase + 8 * v));
        } else {
            const uint4 *p = reinterpret_cast<const uint4 *>(a.words + wbase);
#pragma unroll
            for (int v = 0; v < WPT / 4; v++) {
                uint4 q = __ldg(p + v);
                w[4 * v + 0] = q.x; w[4 * v + 1] = q.y; w[4 * v + 2] = q.z; w[4 * v + 3] = q.w;
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < WPT; j++)
            w[j] = (wbase + j < a.nwords) ? __ldg(a.words + wbase + j) : 0u;
    }
}

template <int WPT, int G, int NP>
__global__ void __launch_bounds__(G * HB_T, 1)
hb_emitf_kernel(hb_stream_args a, uint32_t rshift, uint32_t ntiles_run,
                const uint16_t *__restrict__ subs, const uint64_t *__restrict__ tile_base,
                uint8_t *__restrict__ out, uint64_t out_capacity, uint32_t win, uint32_t stage_bytes,
                uint32_t *__restrict__ status) {
    constexpr int T = HB_T;
    constexpr uint32_t LA = HB_EMITF_LA;
    extern __shared__ __align__(16) uint32_t smem[];
    const uint32_t tab_words = 2u << (a.wf + rshift);
    const uint32_t g = threadIdx.x / T, t = threadIdx.x % T, bar = g + 1u;
    uint32_t *s_grp = smem + tab_words + g * hb_emitf_group_words<WPT>(stage_bytes);
    uint32_t *s_warp = s_grp;                              /* 16 */
    uint32_t *s_w = s_grp + 16;                            /* (WPT + LA) rows of T words */
    uint8_t *s_out = reinterpret_cast<uint8_t *>(s_w + (WPT + LA) * T);   /* staging, 16-aligned */

    const hb_lutref slow{a.lut, a.lut, (1u << a.w1) - 1u};
    {   /* EP-table: every entry from the single-symbol table, R copies side by side */
        const uint32_t R = 1u << rshift;
        uint2 *tab = reinterpret_cast<uint2 *>(smem);
        for (uint32_t x = threadIdx.x; x < (1u << a.wf); x += G * T) {
            uint32_t lo, hi;
            hb_ep_entry(slow, x, a.wf, &lo, &hi);
            for (uint32_t r = 0; r < R; r++) tab[(x << rshift) + r] = make_uint2(lo, hi);
        }
    }
    __syncthreads();
    hb_ptab tb;
    tb.tab = nullptr;
    tb.shift = 3u + rshift;
    tb.mask = ((1u << a.wf) - 1u) << tb.shift;
    tb.saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(smem));
    tb.slow = slow;
    const uint32_t laneoff = (t & ((1u << rshift) - 1u)) << 3;   /* this lane's copy of the table */
    const uint32_t s_out_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_out));
    const uint32_t s_col_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_w) + 4u * t);

    /* software pipeline: the next tile's words, record and output base are fetched as soon as
     * this tile's decode has been issued */
    const uint32_t tstep = gridDim.x * G;
    uint32_t tile = blockIdx.x * G + g, nwin = 0;
    uint32_t w[WPT], wl = 0u;
    uint16_t sub = 0;
    uint64_t B = 0;
    auto fetch = [&](uint32_t tl) {
        const uint64_t tb0 = (uint64_t)tl * (T * WPT);
        hb_load_words_n<WPT>(a, tb0 + (uint64_t)t * WPT, w);
        if (t < LA) wl = tb0 + T * WPT + t < a.nwords ? __ldg(a.words + tb0 + T * WPT + t) : 0u;
        sub = subs[(uint64_t)tl * T + t];
        B = tile_base[tl];
    };
    if (tile < ntiles_run) fetch(tile);
    while (tile < ntiles_run) {
        const uint32_t next = tile + tstep;
        const uint64_t Bt = B;
#pragma unroll
        for (int j = 0; j < WPT; j++) s_w[j * T + t] = w[j];
        if (t > 0) {
#pragma unroll
            for (int j = 0; j < (int)LA; j++) s_w[(WPT + j) * T + t - 1] = w[j];
        }
        if (t < LA) s_w[(WPT + t) * T + T - 1] = wl;
        const uint32_t e = hb_sub_entry(sub), c = hb_sub_count(sub);
        uint32_t nk;
        const uint32_t o = hb_group_exscan(c, s_warp, bar, t, &nk);
        const bool full_out = Bt + nk > out_capacity;
        if (full_out && t == 0) atomicOr(status, HB_ST_OUTPUT_FULL);

        uint32_t lo_b = 0;
        for (uint32_t wb = 0; !full_out && (wb == 0 || wb < nk); wb += win, nwin++) {
            const bool mine = c && o >= wb && o - wb < win;
            const bool last_win = wb + win >= nk;
            const uint32_t al = (uint32_t)((reinterpret_cast<uintptr_t>(out) + Bt + wb) & 15u);
            uint32_t *s_hi = s_warp + 14 + (nwin & 1u);     /* alternating slot: no barrier after the copy-out */
            if (t == 0) {
                /* the previous window's bulk store must have read the staging buffer */
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                *s_hi = nk;                                  /* default: last window */
            }
            hb_group_sync(bar);
            uint32_t fin = 0u, fin_at = 0u;
            if (mine) {
                const uint32_t dst = s_out_saddr + al + (o - wb);
                const uint32_t wend = (dst + c + 3u) & ~3u;
                fin = hb_emit_flat_dev<NP>(tb, laneoff, s_col_saddr, 4u * T, e, dst, dst & 3u, wend);
                fin_at = wend - 4u;
                if (o + c - wb >= win && o + c < nk) *s_hi = o + c;   /* I am the window's last thread */
            }
            if (last_win && next < ntiles_run) fetch(next);
            hb_group_sync(bar);
            /* every in-loop store is done: the final word of each slice once more (its upper
             * lanes are the right neighbour's first bytes, whose own first store zeroed the rest) */
            if (mine) hb_st32((hb_out_t)fin_at, 0u, fin);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            hb_group_sync(bar);
            const uint32_t hi_b = *s_hi;
            if (lo_b < hi_b) {
                uint8_t *gbase = out + Bt + wb - al;          /* 16-byte aligned */
                const uint32_t begb = al + (lo_b - wb), endb = al + (hi_b - wb);
                const uint32_t a0 = (begb + 15u) & ~15u, a1 = endb & ~15u;
                if (a0 < a1) {
                    if (t == 0) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     :: "l"(gbase + a0), "r"(s_out_saddr + a0), "r"(a1 - a0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    if (t >= 32 && t < 64) {                 /* head and tail bytes, one warp */
                        const uint32_t i = t - 32;
                        if (begb + i < a0) gbase[begb + i] = s_out[begb + i];
                        if (a1 + i < endb) gbase[a1 + i] = s_out[a1 + i];
                    }
                } else {
                    for (uint32_t i = begb + t; i < endb; i += T) gbase[i] = s_out[i];   /* < 32 bytes */
                }
            }
            lo_b = hi_b > lo_b ? hi_b : lo_b;
        }
        if (full_out && next < ntiles_run) fetch(next);
        hb_group_sync(bar);       /* the tile's words are dead: the next iteration overwrites them */
        tile = next;
    }
    /* the staging buffer must outlive the last bulk store's reads */
    if (t == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

/* ------------------------------------------------------------------------- */
template <int WPT>
__global__ void __launch_bounds__(HB_T)
hb_emit_kernel(hb_stream_args a, const uint16_t *__restrict__ subs,
               const uint64_t *__restrict__ tile_base, const uint64_t *__restrict__ result, uint8_t *__restrict__ out,
               uint64_t out_capacity, uint32_t win, uint32_t *__restrict__ status) {
    constexpr int T = HB_T;
    constexpr uint32_t S = 32u * WPT;
    constexpr uint32_t TS = T * S;
    __shared__ __align__(16) uint32_t s_fast[1u << HB_WF_MAX];   /* E-table (static: constant address) */
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t *s_warp = smem;                               /* 16 */
    uint8_t *s_out = reinterpret_cast<uint8_t *>(s_warp + 16);   /* staging, 16-aligned */
    const int t = threadIdx.x;

    for (uint32_t i = t; i < (1u << a.wf); i += T) s_fast[i] = __ldg(a.fast + i);
    __syncthreads();
    hb_tables tb;
    tb.fast = s_fast;
    tb.fast_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_fast));
    tb.fmask4 = ((1u << a.wf) - 1u) << 2;
    tb.slow = hb_lutref{a.lut, a.lut, (1u << a.w1) - 1u};
    const uint64_t total_valid = result[0];
    const uint32_t s_out_saddr = hb_opaque((uint32_t)__cvta_generic_to_shared(s_out));

    for (uint32_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        const uint64_t tile_bit0 = (uint64_t)tile * TS;
        const uint64_t sub0 = tile_bit0 + (uint64_t)t * S;
        const uint64_t B = tile_base[tile];
        uint32_t w[WPT + 1];
        hb_load_words<WPT>(a, (uint64_t)tile * (T * WPT) + (uint64_t)t * WPT, w);
        const uint16_t sub = subs[(uint64_t)tile * T + t];   /* already re-chained by the down-sweep kernel */

        const uint32_t e = hb_sub_entry(sub), c = hb_sub_count(sub);
        uint32_t nk;
        const uint32_t o = hb_block_exscan(c, s_warp, &nk);
        const uint32_t lim = sub0 >= a.bits_own ? 0u
                           : (a.bits_own - sub0 < S ? (uint32_t)(a.bits_own - sub0) : S);
        /* symbols past the shard's valid total (a cut-off last codeword) are not written */
        uint32_t nvalid = nk;
        if (B >= total_valid) nvalid = 0;
        else if (B + nk > total_valid) nvalid = (uint32_t)(total_valid - B);
        if (B + nvalid > out_capacity) {
            if (t == 0) atomicOr(status, HB_ST_OUTPUT_FULL);
            __syncthreads();
            continue;
        }

        /* The staging buffer holds `win` bytes of tile output plus one thread's
         * worth of overhang; a tile whose output is larger (data far more
         * compressible than the code table suggests) is emitted in several
         * windows.  Window p takes the threads whose first byte lies in
         * [p*win, (p+1)*win); their slices are contiguous, so it copies out
         * [end of window p-1's threads, end of its own threads). */
        uint32_t lo_b = 0;
        for (uint32_t wb = 0; wb == 0 || wb < nk; wb += win) {
            const bool mine = c && o >= wb && o - wb < win;
            const uint32_t al = (uint32_t)((reinterpret_cast<uintptr_t>(out) + B + wb) & 15u);
            if (t == 0) s_warp[15] = nk;                     /* default: last window */
            __syncthreads();
            if (mine) {
                const hb_out_t dst = (hb_out_t)(s_out_saddr + al + (o - wb));
                if (lim == S) hb_emit_fast<WPT>(tb, w, e, c, dst);
                else hb_emit_slow<WPT>(tb.slow, w, lim, e, c, dst);
                if (o + c - wb >= win && o + c < nk) s_warp[15] = o + c;   /* I am the window's last thread */
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   /* my staging writes -> async proxy */
            __syncthreads();
            uint32_t hi_b = s_warp[15];
            if (hi_b > nvalid) hi_b = nvalid;
            if (lo_b < hi_b) {
                /* staging -> global: s_out[al + (b - wb)] -> out[B + b].  The staging index
                 * is congruent to the global address mod 16, so the 16-byte-aligned middle
                 * goes out as ONE bulk asynchronous copy (TMA, cp.async.bulk) issued by a
                 * single thread; the partial first / last vectors are stored byte-wise. */
                uint8_t *gbase = out + B + wb - al;          /* 16-byte aligned */
                const uint32_t begb = al + (lo_b - wb), endb = al + (hi_b - wb);
                const uint32_t a0 = (begb + 15u) & ~15u, a1 = endb & ~15u;
                if (a0 < a1) {
                    if (t == 0) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     :: "l"(gbase + a0), "r"(s_out_saddr + a0), "r"(a1 - a0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    if (t >= 32 && t < 64) {                 /* head and tail bytes, one warp */
                        const uint32_t i = t - 32;
                        if (begb + i < a0) gbase[begb + i] = s_out[begb + i];
                        if (a1 + i < endb) gbase[a1 + i] = s_out[a1 + i];
                    }
                    if (t == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                } else {
                    for (uint32_t i = begb + t; i < endb; i += T) gbase[i] = s_out[i];   /* < 32 bytes */
                }
            }
            lo_b = hi_b > lo_b ? hi_b : lo_b;
            __syncthreads();
        }
    }
}

#endif /* HB_KERNELS_CUH_ */
