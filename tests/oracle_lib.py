"""ctypes access to the CPU checkers -- TEST INFRASTRUCTURE ONLY.

* ``oracle/liboracle.so``  -- this repo's plain-C restatement (oracle/huff_oracle.c)
* ``oracle/_ref/libref.so`` -- the UNMODIFIED reference CPU sources compiled by
  ``make -C oracle ref`` where the reference is present (absent => the tests compare
  with the reference's recorded results instead, or skip where none are recorded)

Nothing under huffmandecoderongpus_b200/ imports this module.
"""
from __future__ import annotations

import ctypes as C
import functools
import hashlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")
FILES_DIR = os.path.join(REF_DIR, "files")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# SURVEY.md section 8(c): SHA-256 of the reference's own simpleDecode output
# (== the plaintext where it is shipped) and of the .huff input.
CORPORA = {
    # name: (huff file, plaintext file or None, decoded sha256, huff sha256, usize)
    "hello": ("hello.huff", "hello",
              "a591a6d40bf420404a011733cfb7b190d62c65bf0bcda32b57b277d9ad9f146e",
              "bc525ac9a37115c480886c178c7cfd2ad3dbafdd5af38c923f710bb3729ff3e8", 11),
    "paper1": ("paper1.huff", "paper1",
               "8d9c42d9fa58b5bce1a8b5fae3cc27c9eb7cc7a032bc12a633d44e816497e143",
               "bbce832921b1968f88431c4e22a0df7e859cf630d296e637444d2cddf05f5e0a", 53161),
    "news": ("news.huff", "news",
             "7f0482f9774681429eb7021050c17966f6acf19450e170de6611e1ed953d42e8",
             "ff5aab3f9811db808ce3877096daf34830df29732b68198c455e113a46003b0f", 377109),
    "book2": ("book2.huff", "book2",
              "c8538730cf2ce6a243acf3eb299c43d619b5c695d892f4884df796c13081fdf8",
              "50d1826baa8bb7dd2b4be5e421f93e8fc7424ca595f691164d0aaf03a8a26cae", 610856),
    "world192": ("world192.txt.huff", "world192.txt",
                 "1aebdc97d29904b25791da9aa32be90b69d7da6dc0ac9b95512ed27ed40d2112",
                 "b9169e59913ae9167b49d977bf37c3345bee557ce3a6c03bd828577c2de4d01d", 2473400),
    "bible": ("bible.txt.huff", "bible.txt",
              "4e0a7e8dff7d9c82dbded57305c0ca3cdd3c4ca014db27121782fe9710f4723f",
              "3489c852ac8d9e92628d6bade0e5336f5ee0cf2b4b4aa88fea664c99a009f712", 4047392),
    "kjv": ("kjv.txt.huff", None,
            "e4e21579f6360b35e66dc97b67cd732a3f759623e41e4e077bec039eeb79fd0a",
            "1d0e7ce7f8c517e194d65300b99b27026ca39dc7d30e29f82548a7b87b7b485b", 5504597),
    "ecoli": ("E.coli.huff", None,
              "9125dfd87315961ef4286f3856098069e050cc3a2abe65735fe43e69d1996f40",
              "5ce607e6161488db6a14d64b8b80c55e26ebb2fa2a05ab8de6ce63693f68d93d", 4638690),
}


def corpus_path(name: str) -> str | None:
    """Path of a corpus .huff: oracle/_ref/files (all eight, build container
    and GPU box) or tests/golden (the small committed ones)."""
    fn = CORPORA[name][0]
    for d in (FILES_DIR, GOLDEN_DIR):
        p = os.path.join(d, fn)
        if os.path.exists(p):
            return p
    return None


def plaintext_path(name: str) -> str | None:
    fn = CORPORA[name][1] if name in CORPORA else None
    if fn is None:
        return None
    for d in (FILES_DIR, GOLDEN_DIR):
        p = os.path.join(d, fn)
        if os.path.exists(p):
            return p
    return None


def sha256(buf) -> str:
    return hashlib.sha256(memoryview(np.ascontiguousarray(buf))).hexdigest()


# Stand-in streams (not reference data).  The six larger corpora are not part of the
# repository, so the cases that need a large stream also run on streams of the bundled
# generator's models, built on the CPU from a fixed seed; the generated symbols are the
# output a decode must give.  name: (model kind, symbols), sized like the corpora.
STANDIN_SEED = 0x5354414E  # "STAN"
STANDINS = {
    "english4m": (0, 4047392),   # English-like order-0 text, as many symbols as bible.txt
    "dna4m": (2, 4638690),       # four symbols of 2-bit codes, as many as E.coli
    "fib1m": (1, 1 << 20),       # 256 symbols, codes of up to 24 bits
    "uniform1m": (3, 1 << 20),   # eight symbols of 3-bit codes (an odd common length factor)
}


@functools.lru_cache(maxsize=None)
def standin(name: str):
    """(huffmandecoderongpus_b200.HuffFile, generated symbols) of a stand-in stream"""
    import huffmandecoderongpus_b200 as hb
    kind, n = STANDINS[name]
    return hb.Model(kind).huff_file_cpu(STANDIN_SEED, n)


def digest(name: str) -> str:
    """SHA-256 of what decoding a corpus or a stand-in must give"""
    return CORPORA[name][2] if name in CORPORA else sha256(standin(name)[1])


class OraNode(C.Structure):
    _fields_ = [("sym", C.c_uint8), ("izero", C.c_int32), ("ione", C.c_int32)]


class OraStream(C.Structure):
    _fields_ = [("nodes", C.c_int32), ("bits", C.c_uint64), ("usize", C.c_uint64),
                ("tree", C.POINTER(OraNode)), ("data", C.POINTER(C.c_uint8)),
                ("wide", C.c_int)]


NODE_DTYPE = np.dtype([("sym", np.uint8), ("izero", np.int32), ("ione", np.int32)],
                      align=True)
assert NODE_DTYPE.itemsize == 12

_oracle = None


def build_oracle() -> str:
    so = os.path.join(ORACLE_DIR, "liboracle.so")
    src = os.path.join(ORACLE_DIR, "huff_oracle.c")
    if (not os.path.exists(so)) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "liboracle.so"],
                              stdout=subprocess.DEVNULL)
    return so


def oracle():
    global _oracle
    if _oracle is None:
        lib = C.CDLL(build_oracle())
        lib.ora_load_huff.restype = C.POINTER(OraStream)
        lib.ora_load_huff.argtypes = [C.c_char_p]
        lib.ora_free_stream.argtypes = [C.POINTER(OraStream)]
        for f in (lib.ora_tree_height, lib.ora_tree_mindepth, lib.ora_tree_size):
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.c_int]
        lib.ora_simple_decode.restype = C.c_uint64
        lib.ora_simple_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64,
                                          C.c_void_p, C.c_uint64]
        lib.ora_jumptable_decode.restype = C.c_uint64
        lib.ora_jumptable_decode.argtypes = [C.c_void_p, C.c_int, C.c_void_p,
                                             C.c_uint64, C.c_int, C.c_void_p,
                                             C.c_uint64]
        lib.ora_prefix_sizes.restype = None
        lib.ora_prefix_sizes.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64,
                                         C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        lib.ora_pes_decode.restype = C.c_uint64
        lib.ora_pes_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64,
                                       C.c_void_p, C.c_uint64]
        lib.ora_decode_all_bits.restype = None
        lib.ora_decode_all_bits.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64,
                                            C.c_void_p, C.c_void_p]
        _oracle = lib
    return _oracle


class Stream:
    """A loaded .huff stream held in numpy arrays (tree: NODE_DTYPE, data: u8
    with >= 16 zero bytes of padding)."""

    def __init__(self, tree, data, bits, usize):
        self.tree = np.ascontiguousarray(tree, dtype=NODE_DTYPE)
        self.data = np.ascontiguousarray(data, dtype=np.uint8)
        self.bits = int(bits)
        self.usize = int(usize)
        self.nodes = int(self.tree.shape[0])
        assert self.data.size >= (self.bits + 7) // 8 + 16

    @property
    def nbytes(self):
        return (self.bits + 7) // 8


def load_huff(path: str) -> Stream:
    lib = oracle()
    p = lib.ora_load_huff(path.encode())
    if not p:
        raise ValueError(f"oracle could not load {path}")
    s = p.contents
    tree = np.ctypeslib.as_array(C.cast(s.tree, C.POINTER(C.c_uint8)),
                                 shape=(s.nodes * 12,)).copy().view(NODE_DTYPE)
    nbytes = (s.bits + 7) // 8
    data = np.ctypeslib.as_array(s.data, shape=(nbytes + 16,)).copy()
    out = Stream(tree, data, s.bits, s.usize)
    lib.ora_free_stream(p)
    return out


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def simple_decode(st: Stream, bits: int | None = None, cap: int | None = None):
    bits = st.bits if bits is None else bits
    cap = (st.usize if cap is None else cap)
    cap = max(int(cap), bits)  # never overflow even if usize lies
    out = np.zeros(cap + 16, dtype=np.uint8)
    n = oracle().ora_simple_decode(_ptr(st.tree), _ptr(st.data), bits, _ptr(out), cap)
    return out[:n]


def jumptable_decode(st: Stream, jumpbits: int, bits: int | None = None):
    bits = st.bits if bits is None else bits
    cap = max(st.usize, bits)
    out = np.zeros(cap + 16, dtype=np.uint8)
    n = oracle().ora_jumptable_decode(_ptr(st.tree), st.nodes, _ptr(st.data), bits,
                                      jumpbits, _ptr(out), cap)
    if n == 2 ** 64 - 1:
        raise ValueError("jumpbits unsupported for this tree")
    return out[:n]


def pes_decode(st: Stream, bits: int | None = None):
    bits = st.bits if bits is None else bits
    out = np.zeros(bits + 16, dtype=np.uint8)
    n = oracle().ora_pes_decode(_ptr(st.tree), _ptr(st.data), bits, _ptr(out), bits)
    return out[:n]


def prefix_sizes(st: Stream, targetbits: int):
    b = C.c_uint64()
    u = C.c_uint64()
    oracle().ora_prefix_sizes(_ptr(st.tree), _ptr(st.data), targetbits,
                              C.byref(b), C.byref(u))
    return b.value, u.value


def tree_height(st: Stream) -> int:
    return oracle().ora_tree_height(_ptr(st.tree), 0)


def tree_mindepth(st: Stream) -> int:
    return oracle().ora_tree_mindepth(_ptr(st.tree), 0)


# ---- the unmodified reference (32-bit structs, framework/huffdata.h:26-37) ----

class RefCompressed(C.Structure):
    _fields_ = [("bits", C.c_int), ("nodes", C.c_int), ("uncompressedsize", C.c_int),
                ("tree", C.c_void_p), ("data", C.c_void_p)]


class RefUnCompressed(C.Structure):
    _fields_ = [("uncompressedsize", C.c_int), ("data", C.c_void_p)]


_ref = None


def ref():
    """The compiled unmodified reference, or None when oracle/_ref is absent."""
    global _ref
    if _ref is None:
        so = os.path.join(REF_DIR, "libref.so")
        if not os.path.exists(so):
            return None
        lib = C.CDLL(so)
        for name in ("simpleDecode", "jumptableApproach", "pesApproach",
                     "decodeBigtableSimple", "decodeBigtableMultiSym", "linApproach"):
            f = getattr(lib, name)
            f.restype = None
            f.argtypes = [C.POINTER(RefCompressed), C.POINTER(RefUnCompressed), C.c_void_p]
        lib.loadHuffFile.restype = C.POINTER(RefCompressed)
        lib.loadHuffFile.argtypes = [C.c_char_p]
        lib.setTargetSizes.restype = None
        lib.setTargetSizes.argtypes = [C.POINTER(RefCompressed), C.c_int]
        _ref = lib
    return _ref


def ref_decode(st: Stream, approach: str = "simpleDecode", param: int | None = None,
               bits: int | None = None, usize: int | None = None):
    """Run one of the reference's own approaches on st (must fit 32-bit)."""
    lib = ref()
    assert lib is not None
    bits = st.bits if bits is None else bits
    usize = st.usize if usize is None else usize
    assert bits < 2 ** 31
    cd = RefCompressed(bits, st.nodes, usize, st.tree.ctypes.data, st.data.ctypes.data)
    out = np.zeros(max(usize, 1) + 16, dtype=np.uint8)
    ucd = RefUnCompressed(usize, out.ctypes.data)
    if param is None:
        getattr(lib, approach)(C.byref(cd), C.byref(ucd), None)
    else:
        p = C.c_int(param)
        getattr(lib, approach)(C.byref(cd), C.byref(ucd), C.byref(p))
    return out[:usize]


# ---- hand-made codes for tests and probes (not reference code) ----------------
def tree_from_lengths(lengths):
    """canonical-ish complete prefix tree for the given code lengths (Kraft sum 1)"""
    syms = sorted(range(len(lengths)), key=lambda s: (lengths[s], s))
    nodes = [[0, -1, -1]]
    codes = {}
    code, prev = 0, 0
    for s in syms:
        code <<= (lengths[s] - prev)
        prev = lengths[s]
        v = 0
        for i in range(lengths[s] - 1, -1, -1):
            b = (code >> i) & 1
            nxt = nodes[v][1 + b]
            if nxt == -1:
                nodes.append([0, -1, -1])
                nxt = len(nodes) - 1
                nodes[v][1 + b] = nxt
            v = nxt
        nodes[v][0] = s
        codes[s] = [(code >> i) & 1 for i in range(lengths[s] - 1, -1, -1)]
        code += 1
    t = np.zeros(len(nodes), dtype=NODE_DTYPE)
    for i, (sym, a, b) in enumerate(nodes):
        t[i] = (sym & 255, a, b)   # more than 256 leaves: symbols repeat
    return t, codes


def encode_with_codes(codes, syms):
    lens = np.array([len(codes[s]) for s in range(len(codes))])
    total = int(lens[syms].sum())
    bits = np.zeros(total + 64, dtype=np.uint8)
    pos = np.concatenate([[0], np.cumsum(lens[syms])[:-1]])
    maxl = int(lens.max())
    table = np.zeros((len(codes), maxl), dtype=np.uint8)
    for s, c in codes.items():
        table[s, : len(c)] = c
    for k in range(maxl):
        m = lens[syms] > k
        bits[pos[m] + k] = table[syms[m], k]
    data = np.packbits(bits, bitorder="little")
    return np.concatenate([data, np.zeros(32, np.uint8)]), total


def random_lengths(rng, nleaves, maxlen):
    """code lengths of a random complete binary tree with nleaves leaves, depth <= maxlen"""
    lens = [1, 1]
    while len(lens) < nleaves:
        cand = [i for i, l in enumerate(lens) if l < maxlen]
        if not cand:
            break
        # favour deep leaves now and then so that long codewords appear
        i = cand[int(rng.integers(len(cand)))] if rng.random() < 0.7 else max(cand, key=lambda k: lens[k])
        l = lens.pop(i) + 1
        lens += [l, l]
    return lens
