"""CPU emulation of hb_emit32w_kernel's one-window path: chains that end unclipped
(hb_emit_words32_run) and the tail bytes stored again after the warp's barrier.

A lane's last probe may run up to two symbols into its right neighbour's output and complete the
staging word that holds its own last byte; the right neighbour's first store writes that word too,
with zeros in the left lane's bytes.  Both store orders are replayed, for every alignment of the
window in its slice, against the generated symbols.  The records are those of the true chain: the
entry offset of a warp tile's first subsequence is generally not 0 (the offset the down-sweep fix
gives a tile whose hypothesis was wrong)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O
import huffmandecoderongpus_b200 as hb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emul", "emul_run32.cpp")
CSRC = os.path.join(ROOT, "huffmandecoderongpus_b200", "csrc")

_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(tempfile.mkdtemp(prefix="hb_emul_run32_"), "libemul_run32.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC, SRC, "-o", so])
        L = C.CDLL(so)
        L.emul_warp_run32.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p]
        L.emul_warp_run32.restype = C.c_int
        _lib = L
    return _lib


def _stream(lengths, n, seed, skew):
    tree, codes = O.tree_from_lengths(lengths)
    rng = np.random.default_rng(seed)
    w = np.array([2.0 ** (-l) for l in lengths])
    p = w if skew else np.ones(len(lengths))
    syms = rng.choice(len(lengths), size=n, p=p / p.sum())
    data, bits = O.encode_with_codes(codes, syms)
    starts = np.concatenate([[0], np.cumsum(np.asarray(lengths)[syms])[:-1]])
    return tree, syms, data, bits, starts


def _check_warp_tiles(lengths, wpt, n, seed, skew=True, wf=None, tiles=6):
    tree, syms, data, bits, starts = _stream(lengths, n, seed, skew)
    lut = hb.build_lut(tree)
    maxlen = max(lengths)
    if wf is None:
        wf = min(15, maxlen) if maxlen >= 9 else 12
    nb = (bits + 7) // 8
    buf = np.zeros((nb + 3) // 4 * 4 + 64, dtype=np.uint8)
    buf[:nb] = data[:nb]
    words = buf.view("<u4")
    S = 32 * wpt
    nsub = bits // S
    ent = np.ascontiguousarray(lut["entries"], dtype=np.uint32)
    rng = np.random.default_rng(seed + 1)
    firsts = [0] + sorted(int(x) for x in rng.integers(1, nsub - 32, tiles - 1))
    entries = set()
    for s0 in firsts:
        lo = np.searchsorted(starts, np.arange(s0, s0 + 33) * S)
        c = np.diff(lo).astype(np.uint32)
        e = (starts[lo[:32]] - np.arange(s0, s0 + 32) * S).astype(np.uint32)
        assert c.min() >= 8 and e.max() < 32
        entries.add(int(e[0]))
        want = (syms[lo[0]: lo[32]] & 255).astype(np.uint8)
        nk = int(c.sum())
        wl = np.ascontiguousarray(words[s0 * wpt: s0 * wpt + 32 * wpt + 1])
        for al in range(16):
            for order in (0, 1):
                stage = np.full(al + nk + 64, 0xEE, dtype=np.uint8)
                rc = lib().emul_warp_run32(ent.ctypes.data, lut["w1"], wf, wpt, wl.ctypes.data,
                                           e.ctypes.data, c.ctypes.data, al, order, stage.ctypes.data)
                tag = (lengths[:4], wpt, s0, al, order)
                assert rc == 0, tag
                assert np.array_equal(stage[al: al + nk], want), tag
                # only the word holding the last byte may be written past the window
                assert (stage[((al + nk) & ~3) + 4:] == 0xEE).all(), tag
    return entries


@pytest.mark.parametrize("wpt", [8, 4, 16, 2])
@pytest.mark.parametrize("seed", range(3))
def test_random_codes(wpt, seed):
    rng = np.random.default_rng(500 + seed)
    lengths = O.random_lengths(rng, int(rng.choice([64, 200, 256])), int(rng.choice([13, 17, 20])))
    _check_warp_tiles(lengths, wpt, 3 * 32 * 32 * wpt, seed=seed, wf=int(rng.choice([9, 12, 15])))


@pytest.mark.parametrize("wpt", [8, 4])
@pytest.mark.parametrize("lengths", [
    [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 17],    # skewed, up to 17 bits
    [2] * 3 + [4] * 3 + [6] * 3 + [8] * 3 + [10] * 3 + [12] * 3 + [14] * 3 + [16] * 4,
    [5] * 31 + [10] * 32,
])
def test_variable_length_codes(lengths, wpt):
    entries = _check_warp_tiles(lengths, wpt, 3 * 32 * 32 * wpt, seed=sum(lengths) + wpt, tiles=16)
    assert entries - {0}, "no warp tile with a non-zero entry offset"


@pytest.mark.parametrize("wpt", [8, 4])
@pytest.mark.parametrize("lengths", [[2] * 4, [3] * 8, [8] * 256])
def test_fixed_length_codes(lengths, wpt):
    _check_warp_tiles(lengths, wpt, 3 * 32 * 32 * wpt, seed=len(lengths) + wpt, skew=False)


def test_codes_up_to_32_bits():
    # a long-codeword tail: the single-symbol table runs inside the last word too
    lengths = list(range(1, 32)) + [32, 32]
    _check_warp_tiles(lengths, 8, 2 * 32 * 32 * 8, seed=77, wf=12)
