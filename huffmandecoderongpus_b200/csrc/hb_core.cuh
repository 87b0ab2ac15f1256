/*
 * hb_core.cuh -- per-thread decode primitives shared by the sm_100a kernels
 * (hb_kernels.cu) and by the CPU emulation harness used in tests/emul/ to
 * check the tile algorithm without a GPU.  Everything here is plain integer
 * code; HB_HD expands to __host__ __device__ under nvcc and to nothing under
 * a host compiler.
 *
 * Stream semantics (reference framework/mainrun.c:38-55, simpleDecode): bit p
 * of the stream is (data[p/8] >> (p%8)) & 1; bits are consumed root->leaf,
 * 0 -> izero, 1 -> ione.  Read as little-endian 32-bit words, bit p is bit
 * (p & 31) of word p >> 5, so a codeword starting at p is the low bits of the
 * 64-bit window {word[p>>5], word[(p>>5)+1]} shifted right by p & 31.
 */
#ifndef HB_CORE_CUH_
#define HB_CORE_CUH_

#include <stdint.h>

#ifdef __CUDACC__
#define HB_HD __host__ __device__ __forceinline__
#else
#define HB_HD static inline
#endif

#include "hb_format.h"

/* LUT entry (u32):
 *   leaf: bit31 = 0, [7:0] bits consumed at this level (1..width), [15:8] symbol
 *   link: bit31 = 1, [7:0] bits consumed at this level (== this table's width),
 *         [12:8] width of the next table (1..31), [30:13] base index of the
 *         next table inside the same entry array.
 * Level 1 (width w1) lives at index 0 and is staged in shared memory; deeper
 * levels are read from global memory (rare: only codes longer than w1).     */

struct hb_lutref {
    const uint32_t *l1;   /* level-1 table (shared memory on device) */
    const uint32_t *all;  /* whole entry array (global memory on device) */
    uint32_t mask1;       /* (1 << w1) - 1 */
};

HB_HD uint32_t hb_funnel_r(uint32_t lo, uint32_t hi, uint32_t sh) {
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, sh);
#else
    sh &= 31u;
    return sh ? ((lo >> sh) | (hi << (32u - sh))) : lo;
#endif
}

HB_HD uint32_t hb_bit(uint32_t pos) {  /* 1 << (pos & 31) */
    return 1u << (pos & 31u);
}

HB_HD int hb_popc(uint32_t v) {
#ifdef __CUDA_ARCH__
    return __popc(v);
#else
    return __builtin_popcount(v);
#endif
}

/* Decode one codeword whose first bit is bit (pos & 31) of lo; hi is the next
 * stream word.  Returns the codeword length; *sym receives the symbol.       */
HB_HD uint32_t hb_probe(const hb_lutref &lut, uint32_t lo, uint32_t hi,
                        uint32_t pos, uint32_t *sym) {
    uint32_t win = hb_funnel_r(lo, hi, pos);
    uint32_t ent = lut.l1[win & lut.mask1];
    if (ent & HB_LUT_LINK) {
        /* second and deeper levels: 64-bit window, global-memory tables */
        uint64_t w64 = (((uint64_t)hi << 32) | lo) >> (pos & 31u);
        uint32_t used = 0;
        do {
            used += ent & 0xffu;
            uint32_t nw = (ent >> 8) & 31u;
            uint32_t base = (ent >> 13) & 0x3ffffu;
            uint32_t idx = (uint32_t)(w64 >> used) & ((1u << nw) - 1u);
            ent = lut.all[base + idx];
        } while (ent & HB_LUT_LINK);
        *sym = (ent >> 8) & 0xffu;
        return used + (ent & 0xffu);
    }
    *sym = (ent >> 8) & 0xffu;
    return ent & 0xffu;
}

/* ---- tile map entries -----------------------------------------------------
 * A transfer map describes a run of the stream [a, b): for every candidate
 * entry offset e (a true codeword starts at a + e, e < 32) it gives the exit
 * offset x (the first codeword starting at or after b starts at b + x) and
 * the number of codewords that start in [a + e, b).  Packed as
 * (count << 8) | x; tile maps use u32, composed maps u64.                   */

HB_HD uint32_t hb_map_pack32(uint32_t x, uint32_t count) { return (count << 8) | x; }
HB_HD uint64_t hb_map_pack64(uint32_t x, uint64_t count) { return (count << 8) | x; }

/* per-subsequence record written by the sync kernel: entry offset (5 bits) and
 * symbol count (11 bits: at most 512 codewords start in a 512-bit run)        */
HB_HD uint16_t hb_sub_pack(uint32_t e, uint32_t c) { return (uint16_t)((c << 5) | e); }
HB_HD uint32_t hb_sub_entry(uint16_t s) { return s & 31u; }
HB_HD uint32_t hb_sub_count(uint16_t s) { return (uint32_t)s >> 5; }

/* ==== word-granular chain walks =============================================
 * A chain of codewords is followed one 32-bit stream word at a time.  For a
 * word whose first `bound` bit positions may start a codeword (bound = 32
 * except where the stream ends) the walk yields
 *     cnt  = number of codewords of the chain that start in [0, bound)
 *     land = (first codeword start at or after bound) - bound      (0..31)
 * Two chains that land at the same offset behind a word are identical from
 * there on, so "land equals the recorded land" is an exact merge test and the
 * per-word (land, cnt) records are all the state a chain needs.
 *
 * Accumulator convention: acc = (symbols << 8) | position, position relative to
 * the current word (< 32 when a word is entered); table entries add
 * (nsym << 8 | bits) with one instruction (hb_format.h).                      */

struct hb_tables {
    const uint32_t *fast;  /* S- or E-table, 1 << wf entries (host emulation) */
    uint32_t fast_saddr;   /* its shared-state-space address (device) */
    uint32_t fmask4;       /* ((1 << wf) - 1) << 2: byte-offset mask */
    hb_lutref slow;        /* single-symbol multi-level table: long codes, partial words */
};

HB_HD uint32_t hb_funnel_l(uint32_t lo, uint32_t hi, uint32_t sh) {
#ifdef __CUDA_ARCH__
    return __funnelshift_l(lo, hi, sh);
#else
    sh &= 31u;
    return sh ? ((hi << sh) | (lo >> (32u - sh))) : hi;
#endif
}

HB_HD uint32_t hb_ctz(uint32_t v) {   /* v != 0 */
#ifdef __CUDA_ARCH__
    return (uint32_t)__ffs((int)v) - 1u;
#else
    return (uint32_t)__builtin_ctz(v);
#endif
}

HB_HD uint32_t hb_acc_add(uint32_t acc, uint32_t ent) {   /* acc += ent >> 16 */
    return acc + (ent >> 16);
}

/* ent >> 16, written so that the compiler does not fold it with the in-loop
 * accumulate and carry a copy of the accumulator through every iteration */
HB_HD uint32_t hb_hi16(uint32_t ent) {
#ifdef __CUDA_ARCH__
    return __byte_perm(ent, 0u, 0x4432);
#else
    return ent >> 16;
#endif
}

HB_HD uint32_t hb_fast_load(const hb_tables &tb, uint32_t lo2, uint32_t hi2, uint32_t acc) {
    uint32_t x = hb_funnel_r(lo2, hi2, acc) & tb.fmask4;
#ifdef __CUDA_ARCH__
    /* explicit shared-space load: a generic pointer makes the compiler rebuild the
     * shared window base (S2R SR_CgaCtaId ...) on every probe */
    uint32_t ent;
    asm("ld.shared.u32 %0, [%1];" : "=r"(ent) : "r"(x + tb.fast_saddr));
    return ent;
#else
    return *reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(tb.fast) + x);
#endif
}

/* Full word (bound = 32), multi-symbol S-table probes.  acc: in = chain state on
 * entering this word, out = state on entering the next word. */
HB_HD void hb_word_fast(const hb_tables &tb, uint32_t lo, uint32_t hi, uint32_t &acc,
                        uint32_t &land, uint32_t &cnt) {
    const uint32_t lo2 = lo << 2, hi2 = hb_funnel_l(lo, hi, 2);   /* window pre-scaled to byte offsets */
    uint32_t ent, prev;
    for (;;) {
        do {
            ent = hb_fast_load(tb, lo2, hi2, acc);
            acc = hb_acc_add(acc, ent);
        } while (!(acc & 0xE0u));
        prev = acc - hb_hi16(ent);      /* state before the last probe */
        if ((acc & 0xffu) < HB_FAST_MARK) break;
        /* a codeword longer than the table index starts at prev's position */
        uint32_t sym;
        uint32_t len = hb_probe(tb.slow, lo, hi, prev & 0xffu, &sym);
        acc = prev + len + 0x100u;
        ent = 1u;                       /* one start, at offset 0 of the probe */
        if (acc & 0xE0u) break;
    }
    const uint32_t pb = prev & 0xffu;                 /* position of the last probe (< 32) */
    const uint32_t spill = hb_funnel_l(ent & 0xffffu, 0u, pb);   /* its starts at or past bit 32 */
    const uint32_t nsp = (uint32_t)hb_popc(spill);
    const uint32_t pos = (acc & 0xffu) - 32u;
    land = spill ? hb_ctz(spill) : pos;
    cnt = (acc >> 8) - nsp;
    acc = (nsp << 8) | pos;
}

/* Any bound (0..32), one symbol per probe: stream tail and cross-checks. */
HB_HD void hb_word_slow(const hb_lutref &lut, uint32_t lo, uint32_t hi, uint32_t bound,
                        uint32_t &acc, uint32_t &land, uint32_t &cnt) {
    uint32_t pos = acc & 0xffu, n = bound ? acc >> 8 : 0u;   /* carried-in starts lie below the entry position */
    while (pos < bound) {
        uint32_t sym;
        pos += hb_probe(lut, lo, hi, pos, &sym);
        n++;
    }
    land = (pos - bound) & 31u;
    cnt = n;
    acc = pos >= 32u ? pos - 32u : 0u;   /* after a partial word nothing further is owned */
}

HB_HD uint32_t hb_rec_pack(uint32_t land, uint32_t cnt) { return land | (cnt << 5); }
HB_HD uint32_t hb_rec_land(uint32_t r) { return r & 31u; }
HB_HD uint32_t hb_rec_cnt(uint32_t r) { return r >> 5; }

/* bound of word j of a subsequence whose first lim positions are owned */
HB_HD uint32_t hb_bound(uint32_t lim, uint32_t j) {
    return lim >= 32u * (j + 1u) ? 32u : (lim > 32u * j ? lim - 32u * j : 0u);
}

/* multi-symbol probes may carry starts into the next word; that is only exact when word
 * j is fully owned and the next word is fully owned or not owned at all */
HB_HD bool hb_fast_ok(uint32_t lim, uint32_t j) {
    const uint32_t left = lim > 32u * j ? lim - 32u * j : 0u;
    return left >= 64u || left == 32u;
}

/* Chain of entry offset e through a whole subsequence (WPT words, w[WPT] = first
 * word of the next one): fills rec[j] = (land, cnt) per word. */
template <int WPT>
HB_HD void hb_walk(const hb_tables &tb, const uint32_t (&w)[WPT + 1], uint32_t lim, uint32_t e,
                   uint32_t (&rec)[WPT]) {
    uint32_t acc = e;
    if (lim == 32u * WPT) {
#pragma unroll
        for (int j = 0; j < WPT; j++) {
            uint32_t land, cnt;
            hb_word_fast(tb, w[j], w[j + 1], acc, land, cnt);
            rec[j] = hb_rec_pack(land, cnt);
        }
    } else {
        /* partial subsequence (stream tail): multi-symbol probes wherever they are exact
         * (hb_fast_ok), one symbol per probe through the global-memory table elsewhere */
#pragma unroll
        for (int j = 0; j < WPT; j++) {
            uint32_t land, cnt;
            if (hb_fast_ok(lim, j)) hb_word_fast(tb, w[j], w[j + 1], acc, land, cnt);
            else hb_word_slow(tb.slow, w[j], w[j + 1], hb_bound(lim, j), acc, land, cnt);
            rec[j] = hb_rec_pack(land, cnt);
        }
    }
}

/* Re-walk from a new entry offset e, word by word, until the chain lands where
 * the recorded chain landed (identical from there on) or the subsequence ends.
 * rec becomes the chain of e.  Returns true when the landing behind the LAST
 * word changed (the right neighbour's entry offset moves). */
template <int WPT>
HB_HD bool hb_rewalk(const hb_tables &tb, const uint32_t (&w)[WPT + 1], uint32_t lim, uint32_t e,
                     uint32_t (&rec)[WPT]) {
    uint32_t acc = e;
    bool merged = false;
    const bool full = lim == 32u * WPT;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        if (!merged) {
            uint32_t land, cnt;
            if (full || hb_fast_ok(lim, j)) hb_word_fast(tb, w[j], w[j + 1], acc, land, cnt);
            else hb_word_slow(tb.slow, w[j], w[j + 1], hb_bound(lim, j), acc, land, cnt);
            merged = land == hb_rec_land(rec[j]);
            rec[j] = hb_rec_pack(land, cnt);
        }
    }
    return !merged;
}

/* staging-buffer handle: a shared-state-space byte address on the device (a
 * generic pointer would make every store rebuild the shared window base), a
 * plain pointer in the host emulation */
#ifdef __CUDA_ARCH__
typedef uint32_t hb_out_t;
__device__ __forceinline__ void hb_st8(hb_out_t base, uint32_t idx, uint32_t v) {
    asm volatile("st.shared.u8 [%0], %1;" :: "r"(base + idx), "r"(v));
}
#else
typedef uint8_t *hb_out_t;
static inline void hb_st8(hb_out_t base, uint32_t idx, uint32_t v) { base[idx] = (uint8_t)v; }
#endif

/* ==== fixed-length codes (minlen == maxlen == len) ===========================
 * Such codes never self-synchronise (the reference's E.coli corpus: four 2-bit
 * codes), so chains of different entry offsets never merge; but every chain is
 * an arithmetic progression, and entry offsets, counts and exits follow in
 * closed form.  first start at or after bit position p of the chain e, e+len,..: */
HB_HD uint32_t hb_fixed_next(uint32_t e, uint32_t len, uint32_t p) {
    return p <= e ? e : e + ((p - e + len - 1u) / len) * len;
}
/* number of starts of that chain in [lo, hi) */
HB_HD uint32_t hb_fixed_count(uint32_t e, uint32_t len, uint32_t lo, uint32_t hi) {
    const uint32_t a = hb_fixed_next(e, len, lo);
    return a >= hi ? 0u : (hi - a + len - 1u) / len;
}

/* ==== emit walks: decode the chain of entry e and store its symbols ==========
 * E-table probes carry up to two symbols.  The second symbol of the last probe
 * of the LAST word may start in the next subsequence; it is stored only while
 * its index is below c, the chain's symbol count known from the sync kernel. */
template <int WPT>
HB_HD uint32_t hb_emit_fast(const hb_tables &tb, const uint32_t (&w)[WPT + 1], uint32_t e,
                            uint32_t c, hb_out_t out) {
    uint32_t acc = e;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        const uint32_t lo = w[j], hi = w[j + 1];
        const uint32_t lo2 = lo << 2, hi2 = hb_funnel_l(lo, hi, 2);
        uint32_t ent, prev;
        for (;;) {
            do {
                ent = hb_fast_load(tb, lo2, hi2, acc);
                const uint32_t n = acc >> 8;
                hb_st8(out, n, ent);
                /* words before the last: store the second byte unconditionally -- when the
                 * probe held one symbol it is overwritten by the next probe's first store,
                 * which always exists and is this thread's own symbol n + 1 (a probe in
                 * word j < WPT-1 ends at most 63 bits in, i.e. inside word j+1).  Last
                 * word: only a second symbol this thread owns. */
                if (j < WPT - 1) hb_st8(out, n + 1, ent >> 8);
                else { if ((ent & (2u << 24)) && n + 1 < c) hb_st8(out, n + 1, ent >> 8); }
                acc = hb_acc_add(acc, ent);
            } while (!(acc & 0xE0u));
            prev = acc - hb_hi16(ent);
            if ((acc & 0xffu) < HB_FAST_MARK) break;
            uint32_t sym;
            uint32_t len = hb_probe(tb.slow, lo, hi, prev & 0xffu, &sym);
            hb_st8(out, prev >> 8, sym);
            acc = prev + len + 0x100u;
            if (acc & 0xE0u) break;
        }
        acc -= 32u;
    }
    return acc >> 8 < c ? acc >> 8 : c;
}

template <int WPT>
HB_HD uint32_t hb_emit_slow(const hb_lutref &lut, const uint32_t (&w)[WPT + 1], uint32_t lim,
                            uint32_t e, uint32_t c, hb_out_t out) {
    uint32_t pos = e, n = 0;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        const uint32_t limj = lim < 32u * (j + 1) ? lim : 32u * (j + 1);
        while (pos < limj) {
            uint32_t sym;
            pos += hb_probe(lut, w[j], w[j + 1], pos, &sym);
            if (n < c) hb_st8(out, n, sym);
            n++;
        }
    }
    return n < c ? n : c;
}

/* ==== emit walk with word-granular stores ======================================
 * Byte stores into the staging buffer cost ~2.2 shared-memory wavefronts each, and the
 * emit kernel is bound by exactly those.  Here the symbols of a probe are shifted into
 * a 4-byte register window `pend` (newest symbol in the top byte) and a whole 32-bit
 * staging word is stored whenever the running byte count passes a multiple of four.
 *   posk : 8 * (bytes since the 4-byte-aligned address at or below the thread's first
 *          byte) in its low bits.  Bit 5 flips exactly when a staging word completes;
 *          the low 5 bits are the funnel shift that assembles that word from
 *          (new symbols : pend).
 *   The first word a thread stores may start before its slice (lanes below its first
 *   byte hold zeros): those lanes are the LAST bytes of the left neighbour, which every
 *   thread therefore keeps in registers and stores byte-wise after a barrier (the
 *   `tail`).  No other staging byte is written by two threads.
 *   Only probes in the last word can run into the next subsequence; there the symbols
 *   pushed are clipped to the chain's count c.
 * Probes read the E64-table (hb_format.h): LDS.64, up to three symbols.  A 32-bit
 * variant with two symbols per probe was measured slower (0.98 vs 0.78 ms) and dropped. */
struct hb_tables64 {
    const uint32_t *fast;  /* E64-table (host emulation: plain, sc = 3, laneoff = 0) */
    uint32_t fast_saddr;   /* its shared-state-space address (device) */
    uint32_t fmask;        /* byte-offset mask: ((1 << wf) - 1) << sc */
    hb_lutref slow;
    /* device: the table may be held in R = 1 << (sc - 3) copies interleaved entry by entry
     * (copy r of entry x at byte (x << sc) + 8 r); a lane reads copy laneoff / 8, so that
     * lanes of different copies never share a bank and fewer LDS.64 wavefronts are replays */
    uint32_t sc = 3u, laneoff = 0u;
};

/* one probe: symbols (first in the low byte), sel (low 16 bits: PRMT selector for the
 * window update), inc (low 6 bits: 8 * nsym; added to posk as a whole, junk above bit 9),
 * adv (bits consumed, or HB_E64_MARK) */
struct hb_pe { uint32_t syms, sel, inc, adv; };

HB_HD uint32_t hb_prmt(uint32_t a, uint32_t b, uint32_t sel) {
#ifdef __CUDA_ARCH__
    /* raw PRMT: only selector bits 15:0 count and every nibble used here is < 8, so the
     * masking that __byte_perm adds is not needed */
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
#else
    const uint64_t v = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) r |= (uint32_t)((v >> (8u * ((sel >> (4 * i)) & 7u))) & 0xffu) << (8 * i);
    return r;
#endif
}

HB_HD hb_pe hb_probe_words(const hb_tables64 &tb, uint32_t los, uint32_t his, uint32_t acc) {
    const uint32_t x = (hb_funnel_r(los, his, acc) & tb.fmask) | tb.laneoff;
    uint32_t lo, hi;
#ifdef __CUDA_ARCH__
    asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(x + tb.fast_saddr));
#else
    const uint32_t *q = reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(tb.fast) + (x >> (tb.sc - 3u)));
    lo = q[0];
    hi = q[1];
#endif
    hb_pe p;
    p.syms = lo; p.sel = hi; p.inc = hi >> 16; p.adv = hi >> 26;
    return p;
}

/* E64 entry of index x (wf bits, LSB first) from the single-symbol table (hb_format.h; the same
 * values hb_build_tables_kernel writes for the codebook's default width) */
HB_HD void hb_e64_entry(const hb_lutref &slow, uint32_t x, uint32_t wf, uint32_t *lo, uint32_t *hi) {
    uint32_t pos = 0, n = 0, syms = 0;
    while (n < HB_E64_MAXSYM && pos < wf) {
        uint32_t sym;
        const uint32_t len = hb_probe(slow, x >> pos, 0u, 0u, &sym);
        if (pos + len > wf) break;           /* would use bits beyond the index */
        syms |= sym << (8u * n);
        n++;
        pos += len;
    }
    *lo = syms;
    *hi = n ? ((0x3210u + 0x1111u * n) | ((8u * n) << 16) | (pos << 26)) : (0x3210u | (HB_E64_MARK << 26));
}

HB_HD uint32_t hb_pe_nsym(const hb_pe &p) { return (p.inc >> 3) & 7u; }

#ifdef __CUDA_ARCH__
__device__ __forceinline__ void hb_st32(hb_out_t base, uint32_t idx, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" :: "r"(base + idx), "r"(v));
}
#else
static inline void hb_st32(hb_out_t base, uint32_t idx, uint32_t v) {
    for (int i = 0; i < 4; i++) base[idx + i] = (uint8_t)(v >> (8 * i));
}
#endif

/* probe standing for one codeword decoded by the single-symbol table */
HB_HD hb_pe hb_pe_single(const hb_lutref &slow, uint32_t lo, uint32_t hi, uint32_t pos) {
    uint32_t sym;
    const uint32_t len = hb_probe(slow, lo, hi, pos, &sym);
    hb_pe p;
    p.syms = sym; p.sel = 0x4321u; p.inc = 8u; p.adv = len;
    return p;
}

/* the same probe with only its first n symbols (n < its own count) */
HB_HD void hb_pe_clip(hb_pe &p, uint32_t n) {
    p.sel = 0x3210u + 0x1111u * n;
    p.inc = 8u * n;
}

/* keep a loop-invariant value in its register (the compiler otherwise recomputes the
 * pre-scaled window inside the probe loop to save one) */
HB_HD uint32_t hb_keep(uint32_t v) {
#ifdef __CUDA_ARCH__
    asm volatile("" : "+r"(v));
#endif
    return v;
}

/* shift a probe's symbols into the window; store the staging word they complete.  At most
 * four new bytes on top of at most three pending ones: at most one word completes. */
HB_HD uint32_t hb_push(const hb_pe &p, uint32_t &pend, uint32_t posk, hb_out_t &wpp) {
    const uint32_t word = hb_funnel_l(pend, p.syms, posk);   /* pending bytes below the new ones */
    const uint32_t posk_n = posk + p.inc;
    pend = hb_prmt(pend, p.syms, p.sel);
    if ((posk ^ posk_n) & 0x20u) { hb_st32(wpp, 0u, word); wpp += 4; }
    return posk_n;
}

struct hb_tail { hb_out_t at; uint32_t k, bytes; };   /* k bytes (low first) to store at `at` after the barrier */

/* mis: (staging address of out) & 3 */
template <int WPT>
HB_HD hb_tail hb_emit_words(const hb_tables64 &tb, const uint32_t (&w)[WPT + 1], uint32_t e,
                            uint32_t c, hb_out_t out, uint32_t mis) {
    const uint32_t SC = tb.sc;                        /* window pre-scale: log2(bytes per entry and copy set) */
    uint32_t acc = e, pend = 0u, posk = 8u * mis;     /* acc: bit position in the current word */
    hb_out_t wpp = out - mis;                         /* next staging word to store */
#pragma unroll
    for (int j = 0; j < WPT - 1; j++) {
        const uint32_t lo = w[j], hi = w[j + 1];
        const uint32_t los = hb_keep(lo << SC), his = hb_funnel_l(lo, hi, SC);
        for (;;) {
            /* two probes per trip: posk alternates between two registers instead of
             * being copied every probe */
            for (;;) {
                hb_pe p = hb_probe_words(tb, los, his, acc);
                const uint32_t pk2 = hb_push(p, pend, posk, wpp);
                acc += p.adv;
                if (acc & 0xE0u) { posk = pk2; break; }
                p = hb_probe_words(tb, los, his, acc);
                posk = hb_push(p, pend, pk2, wpp);
                acc += p.adv;
                if (acc & 0xE0u) break;
            }
            if (acc < HB_E64_MARK) break;
            /* the last entry was the marker (no symbols): a codeword longer than the table
             * index starts at the position before it */
            acc -= HB_E64_MARK;
            const hb_pe p = hb_pe_single(tb.slow, lo, hi, acc);
            posk = hb_push(p, pend, posk, wpp);
            acc += p.adv;
            if (acc & 0xE0u) break;
        }
        acc -= 32u;
    }
    {   /* last word: the symbols pushed are clipped to c */
        const uint32_t lo = w[WPT - 1], hi = w[WPT];
        const uint32_t los = hb_keep(lo << SC), his = hb_funnel_l(lo, hi, SC);
        uint32_t n = (uint32_t)(wpp - out) + ((posk >> 3) & 3u);   /* symbols pushed so far */
        for (;;) {
            while (!(acc & 0xE0u)) {
                hb_pe p = hb_probe_words(tb, los, his, acc);
                const uint32_t ns = hb_pe_nsym(p);
                if (n + ns > c) hb_pe_clip(p, n < c ? c - n : 0u);
                posk = hb_push(p, pend, posk, wpp);
                n += ns;
                acc += p.adv;
            }
            if (acc < HB_E64_MARK) break;
            acc -= HB_E64_MARK;
            hb_pe p = hb_pe_single(tb.slow, lo, hi, acc);
            if (n >= c) hb_pe_clip(p, 0u);
            posk = hb_push(p, pend, posk, wpp);
            n += 1u;
            acc += p.adv;
            if (acc & 0xE0u) break;   /* a long codeword may end past HB_E64_MARK: not a marker */
        }
    }
    hb_tail tl;
    tl.k = (posk >> 3) & 3u;
    tl.bytes = tl.k ? pend >> ((32u - 8u * tl.k) & 31u) : 0u;
    tl.at = wpp;
    return tl;
}

/* Partial subsequence (stream tail) in the word-store kernel: byte stores, every symbol
 * clipped to the chain's count c -- which is exactly the number of owned codeword starts,
 * so probes may run past the owned bits (into the halo or the zero padding) freely. */
template <int WPT>
HB_HD uint32_t hb_emit_clipped(const hb_tables64 &tb, const uint32_t (&w)[WPT + 1], uint32_t lim,
                               uint32_t e, uint32_t c, hb_out_t out) {
    const uint32_t SC = tb.sc;
    uint32_t acc = e, n = 0u;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        if (32u * j < lim) {
            const uint32_t lo = w[j], hi = w[j + 1];
            const uint32_t los = lo << SC, his = hb_funnel_l(lo, hi, SC);
            for (;;) {
                while (!(acc & 0xE0u)) {
                    const hb_pe p = hb_probe_words(tb, los, his, acc);
                    const uint32_t ns = hb_pe_nsym(p);
#pragma unroll
                    for (uint32_t i = 0; i < HB_E64_MAXSYM; i++)
                        if (i < ns && n + i < c) hb_st8(out, n + i, p.syms >> (8u * i));
                    n += ns;
                    acc += p.adv;
                }
                if (acc < HB_E64_MARK) break;
                acc -= HB_E64_MARK;
                const hb_pe p = hb_pe_single(tb.slow, lo, hi, acc);
                if (n < c) hb_st8(out, n, p.syms);
                n += 1u;
                acc += p.adv;
                if (acc & 0xE0u) break;
            }
            acc -= 32u;
        }
    }
    return n < c ? n : c;
}

HB_HD void hb_store_tail(const hb_tail &tl) {
#pragma unroll
    for (uint32_t i = 0; i < 3u; i++)
        if (i < tl.k) hb_st8(tl.at, i, tl.bytes >> (8u * i));
}

/* ==== emit walk with word-granular stores, 32-bit table entries (hb_emit32_kernel) ==========
 * Same staging discipline as hb_emit_words (register window, whole-word stores, tail after the
 * barrier), but the probes read the E32-table: ONE 32-bit word per index,
 *     [23:0]  first .. third symbol, one byte each (at most HB_E32_MAXSYM)
 *     [25:24] nsym, [31:26] bits consumed; marker (not even one codeword fits): nsym = 0,
 *             bits = HB_E64_MARK
 * An LDS.32 of a warp is one wavefront group of 32 lanes (an LDS.64 is two of 16), and a table of
 * half the size leaves room for twice the copies: measured 2.1 wavefronts per probe against 4.8.
 * No ready-made selector is needed: "shift nsym new bytes into the window" is a funnel shift by
 * 8 * nsym, and the table's top byte, which rides along in the symbol word, is shifted out of
 * every staging word that is stored (a word completes only when at least one byte was pending,
 * because a probe brings at most three).
 * The loops are plain do-while loops with a single exit (one probe per trip): the divergent
 * exits of the two-probe form made every group of lanes run the long-codeword test on its own. */
#define HB_E32_MAXSYM 3
struct hb_tables32 {
    const uint32_t *fast;  /* E32-table (host emulation: plain, sc = 2, lanebase = 0) */
    uint32_t fmask;        /* byte-offset mask: ((1 << wf) - 1) << sc */
    uint32_t lanebase;     /* device: shared address of the table (aligned to its size, so that it can be
                            * OR-ed in) | byte offset of this lane's copy; copies are interleaved entry by
                            * entry (copy r of entry x at byte (x << sc) + 4 r) and sit on disjoint banks */
    hb_lutref slow;
    uint32_t sc, wf;
    uint32_t addbase = 0u; /* device, hb_probe32<true>: the table's address when it cannot be aligned to its size
                            * (128 KB tables); lanebase then holds the copy offset only */
};

/* E32 entry of index x (wf bits, LSB first) from the single-symbol table */
HB_HD uint32_t hb_e32_entry(const hb_lutref &slow, uint32_t x, uint32_t wf) {
    uint32_t pos = 0, n = 0, syms = 0;
    while (n < HB_E32_MAXSYM && pos < wf) {
        uint32_t sym;
        const uint32_t len = hb_probe(slow, x >> pos, 0u, 0u, &sym);
        if (pos + len > wf) break;           /* would use bits beyond the index */
        syms |= sym << (8u * n);
        n++;
        pos += len;
    }
    return n ? (syms | (n << 24) | (pos << 26)) : (HB_E64_MARK << 26);
}

template <bool ADD = false>
HB_HD uint32_t hb_probe32(const hb_tables32 &tb, uint32_t los, uint32_t his, uint32_t acc) {
    const uint32_t x = (hb_funnel_r(los, his, acc) & tb.fmask) | tb.lanebase;
#ifdef __CUDA_ARCH__
    uint32_t ent;
    asm("ld.shared.u32 %0, [%1];" : "=r"(ent) : "r"(ADD ? x + tb.addbase : x));
    return ent;
#else
    return tb.fast[x >> tb.sc];
#endif
}

/* entry standing for one codeword decoded by the single-symbol table.  (A real call instead of nine
 * inlined copies of the multi-level walk shrinks the emit kernel's code by a quarter and was measured
 * 12 % SLOWER: the call's register conventions leak into the hot loops.) */
HB_HD uint32_t hb_e32_single(const hb_lutref &slow, uint32_t lo, uint32_t hi, uint32_t pos) {
    uint32_t sym;
    const uint32_t len = hb_probe(slow, lo, hi, pos, &sym);
    return sym | (1u << 24) | (len << 26);
}

HB_HD uint32_t hb_e32_nsym(uint32_t ent) { return (ent >> 24) & 3u; }
/* 8 * nsym.  (Taking it with IMAD.HI -- a multiply by 2^11 -- to move work from the integer ALU
 * pipe, the kernel's busiest unit, to the FMA pipe was measured slower: 0.665 vs 0.650 ms.) */
HB_HD uint32_t hb_e32_shift(uint32_t ent) { return (ent >> 21) & 0x18u; }
HB_HD uint32_t hb_e32_advance(uint32_t acc, uint32_t ent) { return acc + (ent >> 26); }

/* shift the first t / 8 symbols of ent into the window; store the staging word they complete */
HB_HD uint32_t hb_push32(uint32_t ent, uint32_t t, uint32_t &pend, uint32_t posk, hb_out_t &wpp) {
    const uint32_t word = hb_funnel_l(pend, ent, posk);      /* pending bytes below the new ones */
    const uint32_t posk_n = posk + t;
    pend = hb_funnel_r(pend, ent, t);
    if ((posk ^ posk_n) & 0x20u) { hb_st32(wpp, 0u, word); wpp += 4; }
    return posk_n;
}

/* A chain may be walked in parts of WPT words each (hb_emit32w_kernel's lanes take two consecutive
 * subsequences: their output is contiguous and the chain simply runs on): st carries the position, the
 * register window and the staging pointer from part to part.  `last`: this part ends the lane's chain --
 * only then are the final probes clipped to the count c (of the WHOLE chain). */
struct hb_w32 { uint32_t acc, pend, posk; hb_out_t wpp; };

HB_HD void hb_w32_begin(hb_w32 &st, uint32_t e, hb_out_t out, uint32_t mis) {
    st.acc = e; st.pend = 0u; st.posk = 8u * mis; st.wpp = out - mis;
}

template <int WPT, bool ADD = false>
HB_HD void hb_emit_words32_part(const hb_tables32 &tb, const uint32_t (&w)[WPT + 1], hb_w32 &st,
                                uint32_t c, hb_out_t out, bool last) {
    const uint32_t SC = tb.sc;
    uint32_t acc = st.acc, pend = st.pend, posk = st.posk;
    hb_out_t wpp = st.wpp;
#pragma unroll
    for (int j = 0; j < WPT - 1; j++) {
        const uint32_t lo = w[j], hi = w[j + 1];
        const uint32_t los = hb_keep(lo << SC), his = hb_funnel_l(lo, hi, SC);
        for (;;) {
            do {
                const uint32_t ent = hb_probe32<ADD>(tb, los, his, acc);
                posk = hb_push32(ent, hb_e32_shift(ent), pend, posk, wpp);
                acc = hb_e32_advance(acc, ent);
            } while (!(acc & 0xE0u));
            if (acc < HB_E64_MARK) break;
            /* the last entry was the marker: a codeword longer than the index starts there */
            acc -= HB_E64_MARK;
            const uint32_t ent = hb_e32_single(tb.slow, lo, hi, acc);
            posk = hb_push32(ent, 8u, pend, posk, wpp);
            acc = hb_e32_advance(acc, ent);
            if (acc & 0xE0u) break;
        }
        acc -= 32u;
    }
    {   /* last word.  Probes that start at or below bit 32 - wf end inside the word: all their
         * symbols are this chain's.  Only the one or two probes after that can run into the next
         * subsequence; their symbols are clipped to the chain's count c. */
        const uint32_t lo = w[WPT - 1], hi = w[WPT];
        const uint32_t los = hb_keep(lo << SC), his = hb_funnel_l(lo, hi, SC);
        const uint32_t safe = last ? 32u - tb.wf : 31u;   /* not the last part: no probe is clipped */
        bool done = false;
        for (;;) {
            if (acc <= safe) {
                do {
                    const uint32_t ent = hb_probe32<ADD>(tb, los, his, acc);
                    posk = hb_push32(ent, hb_e32_shift(ent), pend, posk, wpp);
                    acc = hb_e32_advance(acc, ent);
                } while (acc <= safe);
            }
            if (acc < HB_E64_MARK) break;
            acc -= HB_E64_MARK;              /* a long codeword that starts at or below `safe`: ours */
            const uint32_t ent = hb_e32_single(tb.slow, lo, hi, acc);
            posk = hb_push32(ent, 8u, pend, posk, wpp);
            acc = hb_e32_advance(acc, ent);
            if (acc & 0xE0u) { done = true; break; }
        }
        if (!done) {
            uint32_t n = (uint32_t)(wpp - out) + ((posk >> 3) & 3u);   /* symbols pushed so far */
            for (;;) {
                while (!(acc & 0xE0u)) {
                    const uint32_t ent = hb_probe32<ADD>(tb, los, his, acc);
                    const uint32_t ns = hb_e32_nsym(ent);
                    uint32_t t = 8u * ns;
                    if (n + ns > c) t = n < c ? 8u * (c - n) : 0u;
                    posk = hb_push32(ent, t, pend, posk, wpp);
                    n += ns;
                    acc = hb_e32_advance(acc, ent);
                }
                if (acc < HB_E64_MARK) break;
                acc -= HB_E64_MARK;
                const uint32_t ent = hb_e32_single(tb.slow, lo, hi, acc);
                posk = hb_push32(ent, n < c ? 8u : 0u, pend, posk, wpp);
                n += 1u;
                acc = hb_e32_advance(acc, ent);
                if (acc & 0xE0u) break;      /* a long codeword may end past HB_E64_MARK: not a marker */
            }
        }
    }
    if (!last) acc -= 32u;
    st.acc = acc; st.pend = pend; st.posk = posk; st.wpp = wpp;
}

HB_HD hb_tail hb_w32_tail(const hb_w32 &st) {
    hb_tail tl;
    tl.k = (st.posk >> 3) & 3u;
    tl.bytes = tl.k ? st.pend >> ((32u - 8u * tl.k) & 31u) : 0u;
    tl.at = st.wpp;
    return tl;
}

template <int WPT, bool ADD = false>
HB_HD hb_tail hb_emit_words32(const hb_tables32 &tb, const uint32_t (&w)[WPT + 1], uint32_t e,
                              uint32_t c, hb_out_t out, uint32_t mis) {
    hb_w32 st;
    hb_w32_begin(st, e, out, mis);
    hb_emit_words32_part<WPT, ADD>(tb, w, st, c, out, true);
    return hb_w32_tail(st);
}

/* hb_push32 that also keeps the staging word it stores in `last` */
HB_HD uint32_t hb_push32_keep(uint32_t ent, uint32_t t, uint32_t &pend, uint32_t posk, hb_out_t &wpp,
                              uint32_t &last) {
    const uint32_t word = hb_funnel_l(pend, ent, posk);
    const uint32_t posk_n = posk + t;
    pend = hb_funnel_r(pend, ent, t);
    if ((posk ^ posk_n) & 0x20u) { hb_st32(wpp, 0u, word); wpp += 4; last = word; }
    return posk_n;
}

/* Whole chain of a FULL subsequence with an unclipped end (hb_emit32w_kernel's one-window path).
 * The last word runs the plain probe loop until the position leaves the word.  The last probe starts
 * inside the subsequence, so its first codeword is this chain's; the at most HB_E32_MAXSYM - 1 symbols
 * behind it are the right neighbour's first ones, decoded right because the chain is synchronised.
 * Those two bytes can complete at most one staging word: the one holding this chain's last byte, the
 * "boundary word".  The right neighbour's first store writes the same word with zeros where this
 * chain's bytes go, and the two stores land in either order.  So the returned tail holds this chain's
 * k = (out + c) & 3 bytes of the boundary word, to be stored once more after the warp's barrier
 * (hb_store_tail): from the pending bytes, or from the last word stored when the overrun completed the
 * boundary word.  A full subsequence starts at least S / HB_MAX_CODELEN >= 8 codewords, so every
 * chain completes its own first word and no two chains share a boundary word. */
template <int WPT, bool ADD = false>
HB_HD hb_tail hb_emit_words32_run(const hb_tables32 &tb, const uint32_t (&w)[WPT + 1], uint32_t e,
                                  uint32_t c, hb_out_t out, uint32_t mis) {
    const uint32_t SC = tb.sc;
    uint32_t acc = e, pend = 0u, posk = 8u * mis, last = 0u;
    hb_out_t wpp = out - mis;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        const uint32_t lo = w[j], hi = w[j + 1];
        const uint32_t los = hb_keep(lo << SC), his = hb_funnel_l(lo, hi, SC);
        for (;;) {
            do {
                const uint32_t ent = hb_probe32<ADD>(tb, los, his, acc);
                if (j == WPT - 1) posk = hb_push32_keep(ent, hb_e32_shift(ent), pend, posk, wpp, last);
                else posk = hb_push32(ent, hb_e32_shift(ent), pend, posk, wpp);
                acc = hb_e32_advance(acc, ent);
            } while (!(acc & 0xE0u));
            if (acc < HB_E64_MARK) break;
            acc -= HB_E64_MARK;
            const uint32_t ent = hb_e32_single(tb.slow, lo, hi, acc);
            if (j == WPT - 1) posk = hb_push32_keep(ent, 8u, pend, posk, wpp, last);
            else posk = hb_push32(ent, 8u, pend, posk, wpp);
            acc = hb_e32_advance(acc, ent);
            if (acc & 0xE0u) break;
        }
        acc -= 32u;
    }
    /* d: this chain's bytes from the pending word's start, in [-2, 3] (the overrun is at most 2 bytes) */
    const int32_t d = (int32_t)c - (int32_t)(wpp - out);
    const uint32_t np = (posk >> 3) & 3u;
    hb_tail tl;
    if (d >= 0) { tl.k = (uint32_t)d; tl.at = wpp; tl.bytes = pend >> ((32u - 8u * np) & 31u); }
    else { tl.k = (uint32_t)(d + 4); tl.at = wpp - 4; tl.bytes = last; }
    return tl;
}

/* Partial subsequence (stream tail): byte stores, every symbol clipped to the chain's count c */
template <int WPT, bool ADD = false>
HB_HD uint32_t hb_emit_clipped32(const hb_tables32 &tb, const uint32_t (&w)[WPT + 1], uint32_t lim,
                                 uint32_t e, uint32_t c, hb_out_t out) {
    const uint32_t SC = tb.sc;
    uint32_t acc = e, n = 0u;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        if (32u * j < lim) {
            const uint32_t lo = w[j], hi = w[j + 1];
            const uint32_t los = lo << SC, his = hb_funnel_l(lo, hi, SC);
            for (;;) {
                while (!(acc & 0xE0u)) {
                    const uint32_t ent = hb_probe32<ADD>(tb, los, his, acc);
                    const uint32_t ns = hb_e32_nsym(ent);
#pragma unroll
                    for (uint32_t i = 0; i < HB_E32_MAXSYM; i++)
                        if (i < ns && n + i < c) hb_st8(out, n + i, ent >> (8u * i));
                    n += ns;
                    acc = hb_e32_advance(acc, ent);
                }
                if (acc < HB_E64_MARK) break;
                acc -= HB_E64_MARK;
                const uint32_t ent = hb_e32_single(tb.slow, lo, hi, acc);
                if (n < c) hb_st8(out, n, ent);
                n += 1u;
                acc = hb_e32_advance(acc, ent);
                if (acc & 0xE0u) break;
            }
            acc -= 32u;
        }
    }
    return n < c ? n : c;
}

/* ==== flat emit walk (hb_emitf_kernel) =========================================
 * One loop over the whole chain of a subsequence instead of one loop per stream word: the
 * words come from shared memory (a column per thread, so the reads are conflict free) into
 * a 64-bit shifting buffer, the probes read the EP-table (hb_format.h) whose copies keep the
 * lanes of a warp on disjoint banks.
 *   buffer: (hi:lo) holds the next stream bits from bit 0 up and ONE marker bit directly
 *           above them, so "fewer than 32 valid bits" is `hi == 0` and no counter is kept;
 *           a refill ORs the next word in at the marker and moves the marker up 32.
 *   body:   at most one refill, then NP probes of at most wfp bits (NP * wfp <= 32 + the
 *           wfp bits the last probe of a body must still find: NP = 3 for wfp <= 10, else 2).
 *   long codewords (marker entry): consume nothing, so the rest of the body repeats the
 *           same probe; the next body decodes that one codeword with the single-symbol table.
 *   ownership of staging words: a thread stores WHOLE words only -- every word that holds
 *           one of its bytes -- and stops when the word holding its last byte is complete.
 *           The symbols that complete that word are the first ones of the right neighbour's
 *           chain, which this chain simply runs on into.  The first word of a slice may
 *           begin before the slice (those lanes hold zeros); it is the left neighbour's
 *           final word, which every thread therefore returns and stores once more after
 *           the barrier that ends the decode phase.  No symbol is ever clipped. */
struct hb_ptab {
    const uint32_t *tab;   /* plain EP-table, two words per entry (host emulation) */
    uint32_t saddr;        /* device: shared address of the replicated table + this lane's copy */
    uint32_t shift;        /* 3 + rshift */
    uint32_t mask;         /* ((1 << wfp) - 1) << shift */
    hb_lutref slow;
};

/* EP-table entry of index x (wfp bits, LSB first) from the single-symbol table */
HB_HD void hb_ep_entry(const hb_lutref &slow, uint32_t x, uint32_t wfp, uint32_t *lo, uint32_t *hi) {
    uint32_t pos = 0, n = 0, syms = 0;
    while (n < HB_E64_MAXSYM && pos < wfp) {
        uint32_t sym;
        const uint32_t len = hb_probe(slow, x >> pos, 0u, 0u, &sym);
        if (pos + len > wfp) break;          /* would use bits beyond the index */
        syms |= sym << (8u * n);
        n++;
        pos += len;
    }
    *lo = syms;
    *hi = n ? ((0x3210u + 0x1111u * n) | (pos << 16) | ((8u * n) << 21)) : (0x3210u | HB_EP_MARK);
}

HB_HD uint32_t hb_flo(uint32_t v) {   /* index of the highest set bit, v != 0 */
#ifdef __CUDA_ARCH__
    return 31u - (uint32_t)__clz((int)v);
#else
    return 31u - (uint32_t)__builtin_clz(v);
#endif
}

/* Col: next() returns the next stream word of the thread's chain (its own words, then the
 * following subsequences'); e: entry offset; out/mis: first staging byte and its address & 3;
 * wend: end of the last staging word to store.  Returns that last word.
 * This C version is what the CPU emulation runs; the kernel runs hb_emit_flat_dev below, the
 * same loop with its predication written out in PTX. */
template <int NP, class Col>
HB_HD uint32_t hb_emit_flat(const hb_ptab &tb, Col &col, uint32_t e, hb_out_t out, uint32_t mis,
                            hb_out_t wend) {
    const uint32_t w0 = col.next();
    uint32_t lo = hb_funnel_r(w0, 1u, e), hi = e ? 0u : 1u;   /* ((1 << 32) | w0) >> e */
    uint32_t pend = 0u, posk = 8u * mis, word = 0u, m = 0u;
    hb_out_t wpp = out - mis;
    for (;;) {
        if (hi == 0u) {                       /* marker inside lo: fewer than 32 valid bits */
            const uint32_t w = col.next();
            const uint32_t v = hb_flo(lo), mk = 1u << v;
            lo = (lo ^ mk) | (w << v);
            hi = hb_funnel_l(w, 0u, v) | mk;  /* w >> (32 - v), 0 for v == 0 */
        }
        if (m & HB_EP_MARK) {                 /* one codeword longer than the table index */
            uint32_t sym;
            const uint32_t len = hb_probe(tb.slow, lo, hi, 0u, &sym);   /* >= 32 valid bits here */
            word = hb_funnel_l(pend, sym, posk);
            pend = hb_prmt(pend, sym, 0x4321u);
            const uint32_t posk_n = posk + 8u;
            if (len >= 32u) { lo = hi; hi = 0u; }
            else { lo = hb_funnel_r(lo, hi, len); hi >>= len; }
            m = 0u;
            if ((posk ^ posk_n) & 0x20u) {
                hb_st32(wpp, 0u, word);
                wpp += 4;
                if (wpp == wend) return word;
            }
            posk = posk_n;
            continue;
        }
#pragma unroll
        for (int i = 0; i < NP; i++) {
            const uint32_t x = (lo << tb.shift) & tb.mask;
            const uint32_t s = tb.tab[2u * (x >> tb.shift)];
            m = tb.tab[2u * (x >> tb.shift) + 1u];
            const uint32_t m2 = m >> 16;      /* [4:0] bits consumed */
            word = hb_funnel_l(pend, s, posk);
            const uint32_t posk_n = posk + (m >> 21);   /* + 8 * nsym (junk above bit 9) */
            pend = hb_prmt(pend, s, m);
            lo = hb_funnel_r(lo, hi, m2);
            hi = hb_funnel_r(hi, 0u, m2);
            if ((posk ^ posk_n) & 0x20u) {
                hb_st32(wpp, 0u, word);
                wpp += 4;
                if (wpp == wend) return word;
            }
            posk = posk_n;
        }
    }
}

#ifdef __CUDACC__
/* Device version.  cptr/stride: shared address of the thread's column and the byte distance
 * between rows; laneoff: byte offset of this lane's table copy; tb.saddr: the table.
 * Every probe is one straight-line block with two predicated instructions (the staging
 * store and its pointer bump); the refill is one straight-line block predicated on
 * `hi == 0`.  Written in PTX because the compiler turns the C loop above into branches
 * around the store and the refill, which costs more warp instructions than it saves. */
template <int NP>
__device__ __forceinline__ uint32_t hb_emit_flat_dev(const hb_ptab &tb, uint32_t laneoff, uint32_t cptr,
                                                     uint32_t stride, uint32_t e, uint32_t out,
                                                     uint32_t mis, uint32_t wend) {
    uint32_t w0;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(cptr));
    cptr += stride;
    uint32_t lo = __funnelshift_r(w0, 1u, e), hi = e ? 0u : 1u;
    uint32_t pend = 0u, posk = 8u * mis, word = 0u, m = 0u;
    uint32_t wpp = out - mis;
    for (;;) {
        asm volatile("{\n\t"
                     ".reg .pred q;\n\t"
                     ".reg .b32 w, v, mk, t;\n\t"
                     "setp.eq.u32 q, %1, 0;\n\t"
                     "@q ld.shared.u32 w, [%2];\n\t"
                     "@q add.u32 %2, %2, %3;\n\t"
                     "@q bfind.u32 v, %0;\n\t"
                     "@q shl.b32 mk, 1, v;\n\t"
                     "@q shl.b32 t, w, v;\n\t"
                     "@q lop3.b32 %0, %0, mk, t, 0xBE;\n\t"      /* (lo ^ mk) | t */
                     "@q shf.l.wrap.b32 t, w, 0, v;\n\t"         /* w >> (32 - v), 0 for v == 0 */
                     "@q or.b32 %1, t, mk;\n\t"
                     "}"
                     : "+r"(lo), "+r"(hi), "+r"(cptr) : "r"(stride) : "memory");
        if (m & HB_EP_MARK) {                 /* one codeword longer than the table index */
            uint32_t sym;
            const uint32_t len = hb_probe(tb.slow, lo, hi, 0u, &sym);
            word = __funnelshift_l(pend, sym, posk);
            pend = hb_prmt(pend, sym, 0x4321u);
            const uint32_t posk_n = posk + 8u;
            if (len >= 32u) { lo = hi; hi = 0u; }
            else { lo = __funnelshift_r(lo, hi, len); hi >>= len; }
            m = 0u;
            if ((posk ^ posk_n) & 0x20u) {
                asm volatile("st.shared.u32 [%0], %1;" :: "r"(wpp), "r"(word) : "memory");
                wpp += 4;
                if (wpp == wend) return word;
            }
            posk = posk_n;
            continue;
        }
#pragma unroll
        for (int i = 0; i < NP; i++) {
            asm volatile("{\n\t"
                         ".reg .pred p;\n\t"
                         ".reg .b32 t, x, s, m2, pk;\n\t"
                         "shl.b32 t, %0, %8;\n\t"
                         "lop3.b32 x, t, %9, %10, 0xEA;\n\t"     /* (t & mask) | laneoff */
                         "add.u32 x, x, %11;\n\t"
                         "ld.shared.v2.u32 {s, %6}, [x];\n\t"
                         "shr.u32 m2, %6, 16;\n\t"
                         "shf.l.wrap.b32 %5, %2, s, %3;\n\t"     /* staging word: pending bytes below the new ones */
                         "shr.u32 pk, %6, 21;\n\t"
                         "add.u32 pk, pk, %3;\n\t"
                         "prmt.b32 %2, %2, s, %6;\n\t"
                         "shf.r.wrap.b32 %0, %0, %1, m2;\n\t"
                         "shf.r.wrap.b32 %1, %1, 0, m2;\n\t"
                         "xor.b32 t, %3, pk;\n\t"
                         "and.b32 t, t, 32;\n\t"
                         "setp.ne.u32 p, t, 0;\n\t"
                         "@p st.shared.u32 [%4], %5;\n\t"
                         "@p add.u32 %4, %4, 4;\n\t"
                         "mov.b32 %3, pk;\n\t"
                         "}"
                         : "+r"(lo), "+r"(hi), "+r"(pend), "+r"(posk), "+r"(wpp), "+r"(word), "+r"(m)
                         : "r"(0), "r"(tb.shift), "r"(tb.mask), "r"(laneoff), "r"(tb.saddr)
                         : "memory");
            if (wpp == wend) return word;
        }
    }
}
#endif

/* ==== tile-level walks over shared-memory copies ===========================
 * comp: the tile's T*WPT words followed by the first word of the next tile.
 * recs: converged records of the "tile entry offset 0" chain, recs[j*T + t].
 * cs:   exclusive prefix over subsequences of that chain's symbol counts.
 * tile_lim: number of leading bit positions of the tile that are owned.       */

/* Chain of a non-zero tile entry offset e: follow it word by word until it lands
 * where the hypothesis-0 chain landed (exit and remaining count are then those
 * of hypothesis 0) or leaves the tile.  Returns packed (count << 8) | exit. */
template <int WPT, int T>
HB_HD uint32_t hb_hyp_walk(const hb_tables &tb, const uint32_t *comp, const uint32_t *recs,
                           const uint32_t *cs, uint32_t C0, uint32_t X0, uint32_t tile_lim,
                           uint32_t e) {
    uint32_t acc = e, n = 0, land = e;
    const uint32_t nwords = (tile_lim + 31u) >> 5;
    for (uint32_t wi = 0; wi < nwords; wi++) {
        const uint32_t left = tile_lim - 32u * wi;
        const uint32_t bound = left >= 32u ? 32u : left;
        uint32_t cnt;
        /* multi-symbol probes may carry starts into the next word; that is only
         * exact when the next word is fully owned or not owned at all */
        if (left >= 64u || left == 32u) hb_word_fast(tb, comp[wi], comp[wi + 1], acc, land, cnt);
        else hb_word_slow(tb.slow, comp[wi], comp[wi + 1], bound, acc, land, cnt);
        n += cnt;
        const uint32_t t = wi / WPT, j = wi % WPT;
        if (land == hb_rec_land(recs[j * T + t])) {
            uint32_t upto = cs[t];                    /* hypothesis-0 symbols through word wi */
            for (uint32_t jj = 0; jj <= j; jj++) upto += hb_rec_cnt(recs[jj * T + t]);
            return hb_map_pack32(X0 & 31u, n + C0 - upto);
        }
    }
    return hb_map_pack32(land & 31u, n);
}

/* The true entry offset E of a tile differs from the recorded hypothesis (0):
 * redo the (entry, count) records of the leading subsequences until the chain
 * of E enters a subsequence at the offset already on record.  word(i) returns
 * stream word i of the tile (0 past the end of the data); sub points at the
 * tile's T records. */
template <int WPT, int T, class WordFn>
HB_HD void hb_fix_entries(const hb_tables &tb, const WordFn &word, uint16_t *sub,
                          uint32_t tile_lim, uint32_t E) {
    constexpr uint32_t S = 32u * WPT;
    uint32_t e = E;
    for (uint32_t t = 0; t < (uint32_t)T; t++) {
        const uint32_t s0 = t * S;
        if (s0 >= tile_lim) break;
        if (hb_sub_entry(sub[t]) == e) break;
        const uint32_t lim = tile_lim - s0 < S ? tile_lim - s0 : S;
        uint32_t acc = e, n = 0, land = e;
        uint32_t w[WPT + 1];                 /* all words first: independent loads, one round trip */
#pragma unroll
        for (int j = 0; j <= WPT; j++) w[j] = word(t * WPT + j);
#pragma unroll
        for (int j = 0; j < WPT; j++) {
            uint32_t cnt;
            if (lim == S) hb_word_fast(tb, w[j], w[j + 1], acc, land, cnt);
            else hb_word_slow(tb.slow, w[j], w[j + 1], hb_bound(lim, (uint32_t)j), acc, land, cnt);
            n += cnt;
        }
        sub[t] = hb_sub_pack(e, n);
        e = land;
    }
}

/* ==== byte-step transducer walks (sync kernel fast path, full tiles) ==========
 * Table layout in hb_format.h.  A chain is followed 8 bits at a time; its state at
 * a byte boundary is the internal tree node of the unfinished codeword (0 = a
 * codeword starts exactly there), so two chains are identical from a boundary on
 * iff their states there are equal -- an exact merge test with no position
 * arithmetic, no data-dependent trip count and no divergence.  Per 32-bit word the
 * walk records  rec = (state after the word) << 8 | (codewords ENDING in the word).
 *
 * The rest of the pipeline (tile maps, scan, fix, emit) speaks "first codeword START
 * at or after a boundary" and "codewords STARTING in a run".  With d = depth(state)
 * at a boundary b, the unfinished codeword began at b - d, so
 *     forward offset   = length(codeword at b - d) - d          (hb_fsm_fwd)
 *     starts in a run  = ends in it - [d_in > 0] + [d_out > 0].                  */

struct hb_fsm {
    const uint16_t *tab;     /* fsm[state * 256 + byte] (host emulation) */
    uint32_t tab_saddr;      /* its shared-state-space address (device) */
    const uint8_t *depth;    /* fsm_depth[state] */
    const uint16_t *pstep;   /* fsm_pstep[(1 << r) + bits]: root entry for a step of r < 8 bits */
    /* device: the table may be held in R = 1 << lc copies on disjoint banks (hb_fsmc_* below);
     * cbits = this thread's copy index c positioned inside a spread byte, (c << (14 - 2 lc)) * 0x10001 */
    uint32_t lc = 0u, cbits = 0u;
};

/* ---- bank-separated copies of the transducer table --------------------------------------
 * A step's lookup is a random 2-byte read: the 32 lanes of a warp on 32 banks need 3.05
 * wavefronts on average, and the sync kernel is bound by exactly those (87 % of the L1/shared
 * data pipe).  With R copies, each confined to 32 / R banks, only the 32 / R lanes of one copy
 * can collide.  Copy c of entry (state s, byte b) lives at byte
 *     s * (512 R) + (b >> lo) * 128 + c * (128 / R) + (b & mlo) * 2,     lo = 6 - lc, mlo = 2^lo - 1
 * (every 128-byte line holds the same 64 / R entries of all R copies).  The address must stay
 * ONE instruction behind the PRMT that joins state and byte, so every stream word is "spread"
 * once (8 instructions, kept for the re-walks): byte b becomes the 16-bit field
 *     V = (b >> lo) << (14 - lc) | c << (14 - 2 lc) | (b & mlo) << (8 - lc),
 * even bytes of the word in ve, odd bytes in vo.  PRMT then builds X = state << 24 | V << 8 and
 * the address is base + (X >> (15 - lc)) -- a LEA.HI. */
template <int LC>
HB_HD void hb_fsmc_spread(uint32_t w, uint32_t cbits, uint32_t &ve, uint32_t &vo) {
    constexpr uint32_t lo = 6u - LC, mlo = (1u << lo) - 1u, mhi = 0xffu ^ mlo;
    constexpr uint32_t LMe = mlo * 0x00010001u, HMe = mhi * 0x00010001u;
    ve = (w & HMe) * 256u + (w & LMe) * (1u << (8 - LC)) + cbits;      /* multiplies: the FMA pipe is idle */
    vo = (w & (HMe << 8)) | ((w & (LMe << 8)) >> LC) | cbits;
}

/* entry for (state in bits 15:8 of ent, byte I of the spread word) */
template <int LC, int I>
HB_HD uint32_t hb_fsmc_step(const hb_fsm &f, uint32_t ent, uint32_t ve, uint32_t vo) {
    const uint32_t v = (I & 1) ? vo : ve;
#ifdef __CUDA_ARCH__
    const uint32_t x = __byte_perm(ent, v, (I & 2) ? 0x1760 : 0x1540);   /* state : V : (ends) */
    uint16_t r;
    asm("ld.shared.u16 %0, [%1];" : "=h"(r) : "r"(f.tab_saddr + (x >> (15 - LC))));
    return r;
#else
    constexpr uint32_t lo = 6u - LC, mlo = (1u << lo) - 1u;
    const uint32_t vi = (I & 2) ? v >> 16 : v & 0xffffu;
    const uint32_t b = ((vi >> (14 - LC)) << lo) | ((vi >> (8 - LC)) & mlo);
    return f.tab[(ent & 0xff00u) | b];
#endif
}

template <int LC>
HB_HD uint32_t hb_fsmc_word(const hb_fsm &f, uint32_t ve, uint32_t vo, uint32_t &ent) {
    ent = hb_fsmc_step<LC, 0>(f, ent, ve, vo);
    uint32_t acc = ent;
    ent = hb_fsmc_step<LC, 1>(f, ent, ve, vo); acc += ent;
    ent = hb_fsmc_step<LC, 2>(f, ent, ve, vo); acc += ent;
    ent = hb_fsmc_step<LC, 3>(f, ent, ve, vo); acc += ent;
    return (ent & 0xff00u) | (acc & 0xffu);
}

/* v[2 j], v[2 j + 1]: spread word j */
template <int WPT, int LC>
HB_HD void hb_fsmc_walk(const hb_fsm &f, const uint32_t (&v)[2 * WPT], uint32_t state, uint32_t (&rec)[WPT]) {
    uint32_t ent = state << 8;
#pragma unroll
    for (int j = 0; j < WPT; j++) rec[j] = hb_fsmc_word<LC>(f, v[2 * j], v[2 * j + 1], ent);
}

template <int WPT, int LC>
HB_HD bool hb_fsmc_rewalk(const hb_fsm &f, const uint32_t (&v)[2 * WPT], uint32_t state, uint32_t (&rec)[WPT]) {
    uint32_t ent = state << 8;
    bool merged = false;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        if (!merged) {
            const uint32_t r = hb_fsmc_word<LC>(f, v[2 * j], v[2 * j + 1], ent);
            merged = ((r ^ rec[j]) & 0xff00u) == 0u;
            rec[j] = r;
        }
    }
    return !merged;
}

/* entry (state << 8 | byte) in whatever layout the table has: hypothesis lanes only */
HB_HD uint32_t hb_fsm_lookup(const hb_fsm &f, uint32_t sb) {
#ifdef __CUDA_ARCH__
    uint32_t off = 2u * sb;
    if (f.lc) {
        const uint32_t lc = f.lc, lo = 6u - lc, b = sb & 0xffu;
        const uint32_t c = (f.cbits >> (14u - 2u * lc)) & ((1u << lc) - 1u);
        off = ((sb >> 8) << (9u + lc)) + ((b >> lo) << 7) + (c << (7u - lc)) + ((b & ((1u << lo) - 1u)) << 1);
    }
    uint16_t v;
    asm("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(f.tab_saddr + off));
    return v;
#else
    return f.tab[sb];
#endif
}

/* entry for (state in bits 15:8 of ent, byte i of w) */
template <int I>
HB_HD uint32_t hb_fsm_step(const hb_fsm &f, uint32_t ent, uint32_t w) {
#ifdef __CUDA_ARCH__
    /* one PRMT: byte 0 <- byte I of w, byte 1 <- state, bytes 2..3 <- 0 (byte 3 of ent) */
    const uint32_t t = __byte_perm(ent, w, 0x3314 + I);
    uint16_t v;
    asm("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(f.tab_saddr + 2u * t));
    return v;
#else
    return f.tab[(ent & 0xff00u) | ((w >> (8 * I)) & 0xffu)];
#endif
}

/* one stream word: ent in = any value whose bits 15:8 hold the entering state (bits
 * 31:16 zero), out = the last entry read.  Returns the word's record. */
HB_HD uint32_t hb_fsm_word(const hb_fsm &f, uint32_t w, uint32_t &ent) {
    ent = hb_fsm_step<0>(f, ent, w);
    uint32_t acc = ent;
    ent = hb_fsm_step<1>(f, ent, w); acc += ent;
    ent = hb_fsm_step<2>(f, ent, w); acc += ent;
    ent = hb_fsm_step<3>(f, ent, w); acc += ent;
    return (ent & 0xff00u) | (acc & 0xffu);   /* at most 8 ends per byte: the low byte cannot carry */
}

HB_HD uint32_t hb_frec_state(uint32_t r) { return (r >> 8) & 0xffu; }
HB_HD uint32_t hb_frec_ends(uint32_t r) { return r & 0xffu; }

template <int WPT>
HB_HD void hb_fsm_walk(const hb_fsm &f, const uint32_t (&w)[WPT + 1], uint32_t state,
                       uint32_t (&rec)[WPT]) {
    uint32_t ent = state << 8;
#pragma unroll
    for (int j = 0; j < WPT; j++) rec[j] = hb_fsm_word(f, w[j], ent);
}

/* Re-walk from a new entering state until the chain meets the recorded one behind
 * some word (identical from there on) or the subsequence ends; rec becomes the chain
 * of `state`.  Returns true when the state behind the LAST word changed. */
template <int WPT>
HB_HD bool hb_fsm_rewalk(const hb_fsm &f, const uint32_t (&w)[WPT + 1], uint32_t state,
                         uint32_t (&rec)[WPT]) {
    uint32_t ent = state << 8;
    bool merged = false;
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        if (!merged) {
            const uint32_t r = hb_fsm_word(f, w[j], ent);
            merged = ((r ^ rec[j]) & 0xff00u) == 0u;
            rec[j] = r;
        }
    }
    return !merged;
}

/* forward offset of the first codeword start at or after a word boundary whose state
 * has depth d: prev = the word before the boundary, next = the word after it */
HB_HD uint32_t hb_fsm_fwd(const hb_lutref &slow, uint32_t prev, uint32_t next, uint32_t d) {
    if (d == 0u) return 0u;
    uint32_t sym;
    return hb_probe(slow, prev, next, 32u - d, &sym) - d;
}

/* Chain of a non-zero tile entry offset e through a FULL tile (T * WPT words):
 * one partial step to the next byte boundary, byte steps to the next word boundary, then
 * word by word until its state equals the hypothesis-0 chain's recorded state (exit
 * and remaining count are then those of hypothesis 0) or the tile ends.
 * recs[j * T + t]: converged records of hypothesis 0; cs[t]: exclusive prefix over
 * subsequences of its END counts, E0 their total; X0 / d0: its forward exit offset
 * and exit depth.  Returns packed (starts << 8) | exit offset. */
template <int WPT, int T, class WordFn>
HB_HD uint32_t hb_fsm_hyp_walk(const hb_fsm &f, const hb_lutref &slow, const WordFn &word,
                               const uint16_t *recs, const uint32_t *cs, uint32_t E0, uint32_t X0,
                               uint32_t d0, uint32_t e) {
    uint32_t pos = e, n = 0, ent = 0;
    const uint32_t w0 = word(0);
    if (pos & 7u) {
        const uint32_t r = 8u - (pos & 7u);
        ent = f.pstep[(1u << r) + ((w0 >> pos) & ((1u << r) - 1u))];
        n = ent & 0xffu;
        pos += r;
    }
    while (pos & 31u) {
        ent = hb_fsm_lookup(f, (ent & 0xff00u) | ((w0 >> pos) & 0xffu));
        n += ent & 0xffu;
        pos += 8u;
    }
    for (uint32_t wi = 0;;) {           /* pos == 32 * (wi + 1): behind word wi */
        const uint32_t t = wi / WPT, j = wi % WPT;
        if ((((uint32_t)recs[j * T + t] ^ ent) & 0xff00u) == 0u) {
            uint32_t upto = cs[t];      /* hypothesis-0 ends through word wi */
            for (uint32_t jj = 0; jj <= j; jj++) upto += hb_frec_ends(recs[jj * T + t]);
            return hb_map_pack32(X0, n + E0 - upto + (d0 ? 1u : 0u));
        }
        if (++wi == (uint32_t)(T * WPT)) break;
        if (f.lc == 0u) n += hb_frec_ends(hb_fsm_word(f, word(wi), ent));
        else {
            const uint32_t wv = word(wi);
#pragma unroll
            for (int i = 0; i < 4; i++) {
                ent = hb_fsm_lookup(f, (ent & 0xff00u) | ((wv >> (8 * i)) & 0xffu));
                n += ent & 0xffu;
            }
        }
    }
    const uint32_t d = f.depth[hb_frec_state(ent)];
    return hb_map_pack32(hb_fsm_fwd(slow, word(T * WPT - 1), word(T * WPT), d), n + (d ? 1u : 0u));
}

#endif /* HB_CORE_CUH_ */
