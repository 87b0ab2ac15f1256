/*
 * emul_run32.cpp -- TEST INFRASTRUCTURE ONLY: CPU emulation of one warp tile of hb_emit32w_kernel's
 * one-window path (hb_emit_words32_run in hb_core.cuh, shared verbatim with the kernel).
 *
 * 32 lanes each decode one full subsequence into a shared staging slice with whole-word stores and an
 * unclipped end; a lane's overrun may complete the word that holds its last byte, which its right
 * neighbour's first store also writes (with zeros in the left lane's bytes).  The lanes' stores are
 * replayed in a chosen order -- left to right (a right neighbour's first store lands last) or right
 * to left (a left neighbour's overrun lands last) -- then every lane's tail is stored (the kernel does
 * that after a __syncwarp).  tests/test_emul_run32.py checks the slice against the symbols.
 */
#include <stdint.h>
#include <string.h>

#include "hb_core.cuh"

/* lut_entries/w1: single-symbol table; wf: E32 index bits; words: the stream (with one word behind the
 * last subsequence); e/c: the 32 lanes' records (entry offset, codeword starts); al: the window's first
 * byte in the slice (0..15); order: 0 = lanes left to right, 1 = right to left; stage: slice, at least
 * al + sum(c) + 64 bytes, filled by the caller.  Returns 0, or -1 - lane if a tail is not where the
 * lane's bytes end. */
extern "C" int emul_warp_run32(const uint32_t *lut_entries, uint32_t w1, uint32_t wf, int wpt,
                               const uint32_t *words, const uint32_t *e, const uint32_t *c, uint32_t al,
                               int order, uint8_t *stage) {
    hb_lutref slow{lut_entries, lut_entries, (1u << w1) - 1u};
    uint32_t *tab = new uint32_t[(size_t)1 << wf];
    for (uint32_t x = 0; x < (1u << wf); x++) tab[x] = hb_e32_entry(slow, x, wf);
    hb_tables32 tb{tab, ((1u << wf) - 1u) << 2, 0u, slow, 2u, wf};
    uint32_t off[32], o = 0;
    for (int l = 0; l < 32; l++) { off[l] = o; o += c[l]; }
    hb_tail tails[32];
    int rc = 0;
    for (int i = 0; i < 32 && !rc; i++) {
        const int l = order ? 31 - i : i;
        uint8_t *dst = stage + al + off[l];
        const uint32_t mis = (al + off[l]) & 3u;     /* the slice is 16-byte aligned on the device */
        const uint32_t *wl = words + (size_t)l * wpt;
#define RUN(W)                                                                                    \
        if (wpt == W) {                                                                           \
            uint32_t w[W + 1];                                                                    \
            memcpy(w, wl, sizeof(w));                                                             \
            tails[l] = hb_emit_words32_run<W>(tb, w, e[l], c[l], dst, mis);                       \
        }
        RUN(2) RUN(4) RUN(8) RUN(16)
#undef RUN
        if (tails[l].at + tails[l].k != dst + c[l] || tails[l].k > 3u) rc = -1 - l;
    }
    for (int l = 0; l < 32 && !rc; l++) hb_store_tail(tails[l]);
    delete[] tab;
    return rc;
}
