"""Pin the CPU oracle (oracle/huff_oracle.c) before anything trusts it:
golden vector, SHA-256 digests of the reference's own output (SURVEY 8c), and
the unmodified reference compiled into oracle/_ref/libref.so."""
import struct

import numpy as np
import pytest

import oracle_lib as O

ALL = list(O.CORPORA)
SMALL = ["hello", "paper1", "news", "book2"]


def _need(name):
    p = O.corpus_path(name)
    if p is None:
        pytest.skip(f"{name}: corpus not present (run `make -C oracle ref` in the build container)")
    return p


def test_hello_golden_vector():
    # reference framework/mainrun.c:659-663 + files/hello.huff
    st = O.load_huff(_need("hello"))
    assert (st.nodes, st.bits, st.usize) == (15, 32, 11)
    assert bytes(st.data[:4]) == bytes([0x03, 0x65, 0x90, 0xF5])
    bits = "".join(str((st.data[p >> 3] >> (p & 7)) & 1) for p in range(st.bits))
    assert bits == "110" "0000" "01" "01" "001" "100" "0001" "001" "101" "01" "111"
    assert bytes(O.simple_decode(st)) == b"Hello World"
    assert O.tree_height(st) == 4 and O.tree_mindepth(st) == 2


@pytest.mark.parametrize("name", ALL)
def test_header_and_digest(name):
    path = _need(name)
    with open(path, "rb") as f:
        raw = f.read()
    assert O.sha256(np.frombuffer(raw, dtype=np.uint8)) == O.CORPORA[name][3]
    st = O.load_huff(path)
    assert len(raw) == 16 + 9 * st.nodes + st.nbytes  # SURVEY 8: file size identity
    assert st.usize == O.CORPORA[name][4]
    out = O.simple_decode(st)
    assert out.size == st.usize
    assert O.sha256(out) == O.CORPORA[name][2]
    pt = O.plaintext_path(name)
    if pt is not None:
        assert bytes(out) == open(pt, "rb").read()


@pytest.mark.parametrize("name", ALL)
def test_against_unmodified_reference(name):
    """The oracle against the reference's simpleDecode and loadHuffFile: run them where
    oracle/_ref/libref.so is built, else against their recorded results -- the SHA-256 of
    simpleDecode's output (SURVEY 8c) with the shipped plaintext it equals, and the
    big-endian header fields loadHuffFile returns as stored (framework/huffdata.c:27-68)."""
    path = _need(name)
    st = O.load_huff(path)
    got = O.simple_decode(st)
    if O.ref() is not None:
        assert np.array_equal(got, O.ref_decode(st, "simpleDecode"))
        cd = O.ref().loadHuffFile(path.encode()).contents
        header = (cd.bits, cd.nodes, cd.uncompressedsize)
    else:
        assert O.sha256(got) == O.CORPORA[name][2]
        pt = O.plaintext_path(name)
        if pt is not None:
            assert bytes(got) == open(pt, "rb").read()
        with open(path, "rb") as f:
            raw = f.read(16)
        assert raw[:4] == b"HUFF"
        nodes, bits, usize = struct.unpack(">iii", raw[4:16])
        header = (bits, nodes, usize)
    # the reference loader sees the same header
    assert header == (st.bits, st.nodes, st.usize)


@pytest.mark.parametrize("name", ALL)
@pytest.mark.parametrize("jb", [1, 4, 8, 11])
def test_jumptable_matches_serial(name, jb):
    st = O.load_huff(_need(name))
    if jb // O.tree_mindepth(st) > 7 and O.ref() is not None:
        pytest.skip("reference refuses this jumpbits/mindepth")
    want = O.simple_decode(st)
    got = O.jumptable_decode(st, jb)
    assert np.array_equal(got, want)
    if O.ref() is not None and name in SMALL:
        assert np.array_equal(O.ref_decode(st, "jumptableApproach", jb), want)


@pytest.mark.parametrize("name", ["hello", "paper1"])
def test_pes_statement(name):
    st = O.load_huff(_need(name))
    want = O.simple_decode(st)
    assert np.array_equal(O.pes_decode(st), want)
    if O.ref() is not None:
        assert np.array_equal(O.ref_decode(st, "pesApproach"), want)


@pytest.mark.parametrize("name", ["paper1", "news"])
def test_prefix_sizes_match_reference(name):
    st = O.load_huff(_need(name))
    for target in (1, 7, 8, 100, 10000, 12345, st.bits // 2, st.bits - 1):
        b, u = O.prefix_sizes(st, target)
        assert b <= max(target, 1)
        out = O.simple_decode(st, bits=b)
        assert out.size == u
        if O.ref() is not None:
            cd = O.RefCompressed(st.bits, st.nodes, st.usize, st.tree.ctypes.data,
                                 st.data.ctypes.data)
            O.ref().setTargetSizes(O.C.byref(cd), target)
            assert (cd.bits, cd.uncompressedsize) == (b, u)
