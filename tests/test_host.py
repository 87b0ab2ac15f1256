"""Host-side logic and the C-ABI surface, no GPU needed: the shared library loads,
exports every symbol include/*.h (and host/b200approach.h) declares, refuses to
run without a device, and its .huff reader / table builder / generator agree
with the oracle."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import huffmandecoderongpus_b200 as hb

ROOT = O.ROOT


def _declared_functions(header):
    src = open(header).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b((?:hb_|b200)\w+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = hb.lib()
    names = _declared_functions(os.path.join(ROOT, "include", "huffb200.h"))
    names += _declared_functions(os.path.join(ROOT, "huffmandecoderongpus_b200", "host", "b200approach.h"))
    assert len(names) > 30
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(hb.HuffError) as e:
        hb.Context(0)
    assert e.value.code == -1
    # the approach entry point prints and exits, like framework/fastgpu.cu:16-31
    code = ("import sys; sys.path.insert(0, %r); import numpy as np; import huffmandecoderongpus_b200 as hb;"
            "f = hb.HuffFile.load(%r); hb.b200_approach(f.tree, f.data, f.bits, f.usize); print('NOT REACHED')"
            % (ROOT, os.path.join(O.GOLDEN_DIR, "hello.huff")))
    p = subprocess.run(["python", "-c", code], capture_output=True, text=True)
    assert p.returncode != 0 and "NOT REACHED" not in p.stdout
    assert "b200Approach failed" in p.stdout


@pytest.mark.parametrize("name", list(O.CORPORA))
def test_loader_matches_oracle_loader(name):
    p = O.corpus_path(name)
    if p is None:
        pytest.skip("corpus not present")
    a, b = hb.HuffFile.load(p), O.load_huff(p)
    assert (a.nodes, a.bits, a.usize) == (b.nodes, b.bits, b.usize)
    assert np.array_equal(a.tree, b.tree)
    assert np.array_equal(a.data[: a.nbytes], b.data[: b.nbytes])
    assert not a.data[a.nbytes:].any()


def test_container_round_trip_both_widths(tmp_path):
    f = hb.HuffFile.load(os.path.join(O.GOLDEN_DIR, "paper1.huff"))
    for wide in (False, True):
        p = str(tmp_path / f"x{int(wide)}.huff")
        f.save(p, wide=wide)
        raw = open(p, "rb").read()
        assert raw[:4] == (b"HUF8" if wide else b"HUFF")
        assert len(raw) == (24 if wide else 16) + 9 * f.nodes + f.nbytes
        g = hb.HuffFile.load(p)
        assert g.wide == wide and (g.nodes, g.bits, g.usize) == (f.nodes, f.bits, f.usize)
        assert np.array_equal(g.tree, f.tree) and np.array_equal(g.data[: g.nbytes], f.data[: f.nbytes])
        assert np.array_equal(O.load_huff(p).data[: g.nbytes], f.data[: f.nbytes])   # oracle reads HUF8 too
    # the v1 writer is byte-identical to the shipped file
    assert open(str(tmp_path / "x0.huff"), "rb").read() == open(os.path.join(O.GOLDEN_DIR, "paper1.huff"), "rb").read()
    with pytest.raises(hb.HuffError):
        hb.HuffFile.load(os.path.join(O.GOLDEN_DIR, "paper1"))   # plaintext is not a .huff
    with pytest.raises(hb.HuffError):
        hb.HuffFile.load(str(tmp_path / "missing.huff"))


@pytest.mark.parametrize("name", list(O.CORPORA))
def test_lut_decodes_like_the_tree(name):
    """Walk the multi-level table on the CPU (numpy-free loop over a sample of
    offsets) and compare with the oracle's per-offset tree walk (pes.c:30-46)."""
    p = O.corpus_path(name)
    if p is None:
        pytest.skip("corpus not present")
    st = O.load_huff(p)
    lut = hb.build_lut(st.tree)
    assert lut["maxlen"] == O.tree_height(st) and lut["minlen"] == O.tree_mindepth(st)
    ent = lut["entries"]
    nbits = min(st.bits, 20000)
    sym = np.zeros(nbits, np.uint8)
    ln = np.zeros(nbits, np.int32)
    O.oracle().ora_decode_all_bits(st.tree.ctypes.data, st.data.ctypes.data, nbits, sym.ctypes.data, ln.ctypes.data)
    data = st.data
    for b in range(0, nbits - 40, 7):
        win = int.from_bytes(bytes(data[b >> 3:(b >> 3) + 9]), "little") >> (b & 7)
        e = int(ent[win & ((1 << lut["w1"]) - 1)])
        used = 0
        while e & 0x80000000:
            used += e & 0xFF
            nw, base = (e >> 8) & 31, (e >> 13) & 0x3FFFF
            e = int(ent[base + ((win >> used) & ((1 << nw) - 1))])
        assert used + (e & 0xFF) == ln[b] and (e >> 8) & 0xFF == sym[b], (name, b)


def test_malformed_trees_are_rejected():
    f = hb.HuffFile.load(os.path.join(O.GOLDEN_DIR, "hello.huff"))
    t = f.tree.copy(); t["ione"][0] = -1
    with pytest.raises(hb.HuffError) as e:
        hb.build_lut(t)
    assert e.value.code == -2
    t = f.tree.copy(); t["izero"][1] = 0          # cycle back to the root
    with pytest.raises(hb.HuffError):
        hb.build_lut(t)
    t = f.tree.copy(); t["izero"][0] = 999        # child out of range
    with pytest.raises(hb.HuffError):
        hb.build_lut(t)
    with pytest.raises(hb.HuffError):
        hb.build_lut(f.tree[:1])                   # a single node cannot code anything
    # a 40-deep comb: codes longer than 32 bits are refused, not mis-decoded
    n = 2 * 41 + 1
    t = np.zeros(n, dtype=hb.NODE_DTYPE)
    for d in range(41):
        t[2 * d] = (0, 2 * d + 1, 2 * d + 2)
        t[2 * d + 1] = (d, -1, -1)
    t[n - 1] = (99, -1, -1)
    with pytest.raises(hb.HuffError) as e:
        hb.build_lut(t)
    assert e.value.code == -3


def test_models_and_generator():
    eng, fib, dna, u8 = (hb.Model(k) for k in range(4))
    assert eng.nsyms == 63 and eng.maxlen == 17 and eng.minlen == 2   # bible.txt order-0 statistics
    assert fib.nsyms == 256 and 20 < fib.maxlen <= 32
    assert (dna.minlen, dna.maxlen, u8.minlen, u8.maxlen) == (2, 2, 3, 3)
    for m in (eng, fib, dna, u8):
        a = m.symbols_cpu(7, 0, 5000)
        b = m.symbols_cpu(7, 1000, 4000)
        assert np.array_equal(a[1000:], b)      # symbol i depends only on (seed, i)
        assert not np.array_equal(a, m.symbols_cpu(8, 0, 5000))
        data, bits = m.encode_cpu(a)
        st = O.Stream(m.tree, data, bits, a.size)
        assert np.array_equal(O.simple_decode(st), a)
    # the English model reproduces the histogram it was built from
    s = eng.symbols_cpu(1, 0, 400000)
    pt = O.plaintext_path("bible")
    if pt:
        ref = np.bincount(np.fromfile(pt, dtype=np.uint8), minlength=256) / 4047392
        got = np.bincount(s, minlength=256) / s.size
        assert np.abs(ref - got).max() < 0.005


def test_huff_header_promising_more_data_than_the_file_holds(tmp_path):
    """ADVICE r1: an HUF8 header is untrusted -- a bit count the file cannot back (or one that
    would wrap (bits + 7) / 8) is a format error, not a multi-exabyte allocation"""
    import struct
    src = O.corpus_path("hello")
    raw = open(src, "rb").read()
    nodes = struct.unpack(">i", raw[4:8])[0]
    body = raw[16: 16 + 9 * nodes]
    for bits in (2 ** 64 - 3, 2 ** 40, 8 * 5):   # hello holds 4 data bytes
        p = tmp_path / f"bad{bits}.huff"
        p.write_bytes(b"HUF8" + struct.pack(">i", nodes) + struct.pack(">QQ", bits, 11) + body + raw[16 + 9 * nodes:])
        with pytest.raises(hb.HuffError) as e:
            hb.HuffFile.load(str(p))
        assert e.value.code == -8
