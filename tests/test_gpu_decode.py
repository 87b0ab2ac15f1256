"""Parity tests proper: the sm_100a kernels, called through the C ABI
(libhuffb200.so), against the CPU oracle, the reference's SHA-256 digests and
size-independent properties (encode -> decode round trips at full size).
Run with `pytest -m gpu` on a B200."""
import numpy as np
import pytest

import oracle_lib as O
import huffmandecoderongpus_b200 as hb

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SEED = 0x48554646  # "HUFF"


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "these tests need a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(0)
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ctx(dev):
    c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream)
    yield c
    c.close()


def _stream(name):
    if name in O.STANDINS:
        return O.standin(name)[0]
    p = O.corpus_path(name)
    if p is None:
        pytest.skip(f"{name} corpus not present")
    return hb.HuffFile.load(p)


def _large_text():
    """kjv where the corpus is present, else the English-like stand-in of about the same size"""
    return "kjv" if O.corpus_path("kjv") is not None else "english4m"


def _to_dev(data: np.ndarray, nbytes: int, dev, extra=0):
    """compressed bytes -> CUDA uint8 tensor, zero padded to a multiple of 16"""
    n = (nbytes + 15) // 16 * 16 + 16 + extra
    t = torch.zeros(n, dtype=torch.uint8, device=dev)
    t[:nbytes] = torch.from_numpy(np.ascontiguousarray(data[:nbytes])).to(dev)
    return t


def _decode_dev(ctx, cb, f, dev, bits=None, cap=None, out_offset=0):
    bits = f.bits if bits is None else bits
    comp = _to_dev(f.data, (bits + 7) // 8, dev)
    cap = (f.usize if cap is None else cap)
    raw = torch.zeros(cap + 64 + out_offset, dtype=torch.uint8, device=dev)
    out = raw[out_offset:]
    res = hb.decode_device(ctx, cb, comp.data_ptr(), comp.numel(), bits, out.data_ptr(), cap)
    return out[: res["n_symbols"]].cpu().numpy(), res, raw


@pytest.mark.parametrize("name", list(O.CORPORA) + list(O.STANDINS))
def test_corpora_host_buffers(ctx, name):
    """BASELINE configs 1-3: every shipped corpus through hb_decode_host (upload,
    decode, download), byte-exact against the reference's own output digest; the
    stand-in streams against their generated symbols."""
    f = _stream(name)
    out = np.zeros(f.usize + 3, dtype=np.uint8)
    res = hb.decode_host(ctx, f.tree, f.data, f.bits, out[: f.usize])
    assert res["n_symbols"] == f.usize
    if name in O.CORPORA:
        assert f.usize == O.CORPORA[name][4]
    assert O.sha256(out[: f.usize]) == O.digest(name)
    assert res["launches"] > 0 and res["ms_total"] > 0
    pt = O.plaintext_path(name)
    if pt is not None:
        assert bytes(out[: f.usize]) == open(pt, "rb").read()


@pytest.mark.parametrize("name,chunk", [("kjv", 64 << 10), ("kjv", 1 << 20), ("ecoli", 200000),
                                        ("world192", 8192), ("paper1", 8192),
                                        ("english4m", 64 << 10), ("english4m", 1 << 20), ("dna4m", 200000),
                                        ("fib1m", 8192), ("uniform1m", 8192)])
def test_host_path_pipelined_chunks(dev, name, chunk):
    """hb_decode_host on streams longer than two chunks: byte-range chunks on one
    GPU with overlapped upload / decode / download, pinned and pageable buffers."""
    f = _stream(name)
    c = hb.Context(0)
    c.set_host_chunk(chunk)
    for pinned in (False, True):
        if pinned:
            hc = torch.zeros(f.data.size, dtype=torch.uint8).pin_memory()
            hc.copy_(torch.from_numpy(f.data))
            ho = torch.zeros(f.usize + 16, dtype=torch.uint8).pin_memory()
            data, out = hc.numpy(), ho.numpy()
        else:
            data, out = f.data, np.zeros(f.usize + 16, dtype=np.uint8)
        res = hb.decode_host(c, f.tree, data, f.bits, out[: f.usize])
        assert res["n_symbols"] == f.usize
        assert O.sha256(out[: f.usize]) == O.digest(name)
        assert not out[f.usize:].any()
    with pytest.raises(hb.HuffError) as e:
        hb.decode_host(c, f.tree, f.data, f.bits, np.zeros(f.usize - 1, dtype=np.uint8))
    assert e.value.code == -6
    c.close()


def test_host_path_pipelined_short_last_chunk_and_cut_codeword(dev):
    """ADVICE r1: a last chunk shorter than the 16-byte halo -- the last-but-one chunk must not
    count bits (nor read bytes) past the end of the stream.  The stream is also cut inside a
    codeword and decoded twice into a context whose cached device buffer holds the bytes of a
    LONGER earlier decode behind the new end: the cut-off codeword must emit nothing."""
    f = _stream(_large_text())
    st = O.Stream(f.tree, f.data, f.bits, f.usize)
    chunk = 65536
    c = hb.Context(0)
    c.set_host_chunk(chunk)
    out = np.zeros(f.usize + 16, dtype=np.uint8)
    hb.decode_host(c, f.tree, f.data, f.bits, out[: f.usize])          # fills the cached buffers
    for tail_bytes in (1, 7, 15):
        for cut in (0, 3):
            nbytes = 30 * chunk + tail_bytes
            bits = 8 * nbytes - cut
            want = O.simple_decode(st, bits=bits)
            for _ in range(2):
                out[:] = 0
                res = hb.decode_host(c, f.tree, f.data[: nbytes + 8].copy(), bits, out[: want.size])
                assert res["n_symbols"] == want.size, (tail_bytes, cut)
                assert np.array_equal(out[: want.size], want), (tail_bytes, cut)
    c.close()


def test_shard_host_halves_match_oracle(dev):
    """hb_shard_map_host / hb_shard_emit_host: the rank-local halves with host buffers, here for
    two shards decoded one after the other on one GPU (the exchange done by hand)"""
    name = _large_text()
    f = _stream(name)
    c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream)
    cb = hb.Codebook(c, f.tree)
    nbytes = f.nbytes
    per = (nbytes // 2) // 16 * 16
    maps = torch.zeros(64, dtype=torch.int64, device=dev)
    eb = torch.zeros(4, dtype=torch.int64, device=dev)
    outs = []
    geo = []
    for r in range(2):
        a = r * per
        b = nbytes if r == 1 else per
        halo = min(nbytes, b + 16)
        own = f.bits - 8 * a if r == 1 else 8 * (b - a)
        avail = own if r == 1 else min(f.bits - 8 * a, 8 * (halo - a))
        geo.append((a, halo, own, avail))
    # pass 1: both maps (a real run has one rank per shard; here the second map overwrites the
    # context's state, so shard 0 is mapped again before its emit)
    for r in (0, 1):
        a, halo, own, avail = geo[r]
        hb.shard_map_host(c, cb, f.data[a:halo].copy(), halo - a, own, avail, maps[32 * r:].data_ptr())
    for r in (0, 1):
        a, halo, own, avail = geo[r]
        hb.shard_map_host(c, cb, f.data[a:halo].copy(), halo - a, own, avail, 0)
        hb.shard_compose(c, maps.data_ptr(), 2, r, eb.data_ptr())
        h_out = np.zeros(f.usize, dtype=np.uint8)
        res = hb.shard_emit_host(c, cb, eb.data_ptr(), h_out)
        outs.append(h_out[: res["n_symbols"]].copy())
        assert res["out_base"] == (0 if r == 0 else outs[0].size)
    got = np.concatenate(outs)
    assert got.size == f.usize and O.sha256(got) == O.digest(name)
    cb.close()
    c.close()


@pytest.mark.parametrize("name", ["hello", "paper1", "news", "book2", "kjv", "english4m", "dna4m"])
def test_approach_drop_in(name):
    """The bigtable suite (framework/mainrun.c:541-588) calling convention:
    reference-layout structs, zeroed usize+3 output, 1 checked + repeated runs
    (framework/decodeUtil.c:30-70)."""
    f = _stream(name)
    st = O.Stream(f.tree, f.data, f.bits, f.usize)
    want = O.simple_decode(st)
    for rep in range(3):
        got = hb.b200_approach(f.tree, f.data, f.bits, f.usize)
        assert np.array_equal(got, want)
    assert hb.lib().b200ApproachLastSymbols() == f.usize
    assert hb.lib().b200ApproachLastDeviceMs() > 0


@pytest.mark.parametrize("wpt", [4, 8, 16])
@pytest.mark.parametrize("name", ["hello", "paper1", "world192", "kjv", "ecoli", "english4m", "dna4m", "fib1m", "uniform1m"])
def test_device_resident_all_shapes(dev, name, wpt):
    f = _stream(name)
    c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream, words_per_thread=wpt)
    cb = hb.Codebook(c, f.tree)
    got, res, _ = _decode_dev(c, cb, f, dev)
    assert got.size == f.usize and O.sha256(got) == O.digest(name)
    cb.close()
    c.close()


def test_prefix_sweep(ctx, dev):
    # reference graphtest / setTargetSizes, framework/mainrun.c:361-410
    f = _stream("paper1")
    st = O.Stream(f.tree, f.data, f.bits, f.usize)
    cb = hb.Codebook(ctx, f.tree)
    for target in list(range(1, 40)) + list(range(10000, f.bits, 31337)) + [f.bits - 1, f.bits]:
        bits, usize = O.prefix_sizes(st, target)
        got, res, _ = _decode_dev(ctx, cb, f, dev, bits=bits, cap=usize)
        assert res["n_symbols"] == usize, target
        assert np.array_equal(got, O.simple_decode(st, bits=bits)), target


def test_cut_inside_codeword_and_empty(ctx, dev):
    f = _stream("paper1")
    st = O.Stream(f.tree, f.data, f.bits, f.usize)
    cb = hb.Codebook(ctx, f.tree)
    for bits in [0, 1, 2, 3, 31, 32, 33, 127, 128, 129, 4095, 4096, 4097, 32767, 32768, 32769, 100001]:
        want = O.simple_decode(st, bits=bits)
        got, res, _ = _decode_dev(ctx, cb, f, dev, bits=bits, cap=want.size + 8)
        assert res["n_symbols"] == want.size and np.array_equal(got, want), bits


def test_output_alignment_and_no_overrun(ctx, dev):
    f = _stream("paper1")
    want = O.simple_decode(O.Stream(f.tree, f.data, f.bits, f.usize))
    cb = hb.Codebook(ctx, f.tree)
    for off in (0, 1, 3, 7, 8, 15):
        got, res, raw = _decode_dev(ctx, cb, f, dev, out_offset=off)
        assert np.array_equal(got, want)
        host = raw.cpu().numpy()
        assert not host[:off].any() and not host[off + want.size:].any()


def test_output_too_small_and_bad_args(ctx, dev):
    f = _stream("paper1")
    cb = hb.Codebook(ctx, f.tree)
    with pytest.raises(hb.HuffError) as e:
        _decode_dev(ctx, cb, f, dev, cap=f.usize - 1)
    assert e.value.code == -6
    comp = _to_dev(f.data, f.nbytes, dev, extra=16)
    out = torch.zeros(f.usize + 64, dtype=torch.uint8, device=dev)
    with pytest.raises(hb.HuffError) as e:   # misaligned compressed pointer
        hb.decode_device(ctx, cb, comp.data_ptr() + 4, comp.numel() - 4, f.bits, out.data_ptr(), f.usize)
    assert e.value.code == -4
    with pytest.raises(hb.HuffError) as e:   # fewer readable bytes than the stream needs
        hb.decode_device(ctx, cb, comp.data_ptr(), f.nbytes - 1, f.bits, out.data_ptr(), f.usize)
    assert e.value.code == -4
    bad = f.tree.copy()
    bad["ione"][0] = -1                      # half-leaf root
    with pytest.raises(hb.HuffError) as e:
        hb.Codebook(ctx, bad)
    assert e.value.code == -2


@pytest.mark.parametrize("path", ["words32w", "words32w1", "words64w", "words32", "words"])
def test_word_store_kernels_edge_cases(dev, path):
    """The word-store emit kernels on the cases that exercise their end-of-stream bookkeeping (forced
    here: the automatic choice uses them for large streams only): streams cut inside a codeword and at
    every position around word / subsequence / tile boundaries, every output alignment with nothing
    written outside the slice, an output buffer that is too small or exactly large enough."""
    f = _stream("paper1")
    st = O.Stream(f.tree, f.data, f.bits, f.usize)
    c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream)
    if path == "words32w1":
        c.set_emit_lane_subsequences(1)
        path = "words32w"
    c.set_emit_path(path)
    cb = hb.Codebook(c, f.tree)
    for bits in [0, 1, 2, 3, 31, 32, 33, 255, 256, 257, 511, 512, 513, 8191, 8192, 8193, 65535, 65536, 65537, 100001, f.bits - 1]:
        want = O.simple_decode(st, bits=bits)
        got, res, _ = _decode_dev(c, cb, f, dev, bits=bits, cap=want.size + 8)
        assert res["n_symbols"] == want.size and np.array_equal(got, want), bits
    want = O.simple_decode(st)
    for off in (0, 1, 3, 7, 8, 15):
        got, res, raw = _decode_dev(c, cb, f, dev, out_offset=off)
        host = raw.cpu().numpy()
        assert np.array_equal(got, want) and not host[:off].any() and not host[off + want.size:].any()
    got, res, _ = _decode_dev(c, cb, f, dev, cap=f.usize)            # exactly large enough
    assert res["n_symbols"] == f.usize and np.array_equal(got, want)
    for short in (1, 17, 5000):
        with pytest.raises(hb.HuffError) as e:
            _decode_dev(c, cb, f, dev, cap=f.usize - short)
        assert e.value.code == -6
    got, res, _ = _decode_dev(c, cb, f, dev)                         # the context still works afterwards
    assert np.array_equal(got, want)
    cb.close()
    c.close()


@pytest.mark.parametrize("name,nshards,path", [("paper1", 3, "auto"), ("kjv", 2, "auto"), ("kjv", 8, "auto"),
                                               ("ecoli", 4, "auto"), ("kjv", 3, "words32w"), ("paper1", 2, "words32w"),
                                               ("kjv", 2, "words32"), ("english4m", 2, "auto"), ("english4m", 8, "auto"),
                                               ("dna4m", 4, "auto"), ("english4m", 3, "words32w"), ("english4m", 2, "words32"),
                                               ("fib1m", 5, "auto"), ("uniform1m", 3, "auto")])
def test_byte_range_shards_on_one_gpu(dev, name, nshards, path):
    """The multi-GPU decomposition with every 'rank' run on cuda:0: one context
    per rank, maps gathered by concatenation, hb_shard_compose, independent emit."""
    f = _stream(name)
    want = O.simple_decode(O.Stream(f.tree, f.data, f.bits, f.usize))
    per = (f.nbytes // nshards) // 16 * 16
    bounds = [r * per for r in range(nshards)] + [f.nbytes]
    stream = torch.cuda.current_stream().cuda_stream
    ctxs = [hb.Context(0, stream=stream) for _ in range(nshards)]
    for c in ctxs:
        c.set_emit_path(path)
    cbs = [hb.Codebook(c, f.tree) for c in ctxs]
    all_maps = torch.zeros(nshards * 32, dtype=torch.int64, device=dev)
    shards = []
    for r in range(nshards):
        a, b = bounds[r], bounds[r + 1]
        last = r == nshards - 1
        bits_own = f.bits - 8 * a if last else 8 * (b - a)
        halo_end = min(f.nbytes, b + 16)
        bits_avail = bits_own if last else min(f.bits - 8 * a, 8 * (halo_end - a))
        comp = _to_dev(f.data[a:], halo_end - a, dev)
        shards.append((comp, bits_own, bits_avail))
        hb.shard_map(ctxs[r], cbs[r], comp.data_ptr(), comp.numel(), bits_own, bits_avail,
                     all_maps[r * 32:].data_ptr())
    pieces, base_expect = [], 0
    for r, (comp, bo, ba) in enumerate(shards):
        eb = torch.zeros(4, dtype=torch.int64, device=dev)
        hb.shard_compose(ctxs[r], all_maps.data_ptr(), nshards, r, eb.data_ptr())
        out = torch.zeros(want.size + 64, dtype=torch.uint8, device=dev)
        res = hb.shard_emit(ctxs[r], cbs[r], comp.data_ptr(), comp.numel(), bo, ba, eb.data_ptr(),
                            out.data_ptr(), want.size)
        # each rank writes its own slice starting at 0; out_base says where it belongs
        assert res["out_base"] == base_expect
        assert int(eb[2]) == want.size
        base_expect += res["n_symbols"]
        pieces.append(out[: res["n_symbols"]].cpu().numpy())
    got = np.concatenate(pieces)
    assert got.size == want.size and np.array_equal(got, want)
    for cb in cbs:
        cb.close()
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("kind,n", [(hb.MODEL_ENGLISH, 1 << 20), (hb.MODEL_FIBONACCI, 1 << 20),
                                    (hb.MODEL_DNA, 1 << 18), (hb.MODEL_UNIFORM8, 1 << 15)])
def test_gpu_encoder_matches_cpu_encoder_and_oracle(ctx, dev, kind, n):
    """The bundled generator: GPU-built stream == CPU-built stream bit for bit, the
    oracle decodes it back to the generated symbols, and so does the GPU decoder."""
    m = hb.Model(kind)
    f, syms = m.huff_file_cpu(SEED, n)
    comp = torch.zeros((f.nbytes + 15) // 16 * 16 + 32, dtype=torch.uint8, device=dev)
    bits = hb.gen_encode_device(ctx, m, SEED, 0, n, comp.data_ptr(), comp.numel())
    assert bits == f.bits == hb.gen_count_bits_device(ctx, m, SEED, 0, n)
    assert np.array_equal(comp[: f.nbytes].cpu().numpy(), f.data[: f.nbytes])
    assert np.array_equal(O.simple_decode(O.Stream(f.tree, f.data, f.bits, f.usize)), syms)
    cb = hb.Codebook(ctx, m.tree)
    out = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
    res = hb.decode_device(ctx, cb, comp.data_ptr(), comp.numel(), bits, out.data_ptr(), n)
    assert res["n_symbols"] == n
    assert np.array_equal(out[:n].cpu().numpy(), syms)
    assert hb.gen_verify_device(ctx, m, SEED, 0, n, out.data_ptr()) == 0
    out[n // 2] ^= 1
    assert hb.gen_verify_device(ctx, m, SEED, 0, n, out.data_ptr()) == 1


@pytest.mark.parametrize("kind,log2n,wpt", [(hb.MODEL_ENGLISH, 30, 4), (hb.MODEL_ENGLISH, 30, 8),
                                            (hb.MODEL_FIBONACCI, 30, 4), (hb.MODEL_FIBONACCI, 32, 8)])
def test_full_size_round_trip(dev, kind, log2n, wpt):
    """BASELINE configs 4/5 at full single-GPU size: generate + encode on the
    device (> 2^31 bits: the 64-bit path), decode, and compare every byte with
    the regenerated symbols; the CPU oracle checks a prefix."""
    n = 1 << log2n
    c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream, words_per_thread=wpt)
    m = hb.Model(kind)
    bits = hb.gen_count_bits_device(c, m, SEED, 0, n)
    assert bits > 2 ** 31
    nbytes = (bits + 7) // 8
    comp = torch.zeros((nbytes + 15) // 16 * 16 + 32, dtype=torch.uint8, device=dev)
    assert hb.gen_encode_device(c, m, SEED, 0, n, comp.data_ptr(), comp.numel()) == bits
    cb = hb.Codebook(c, m.tree)
    out = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
    res = hb.decode_device(c, cb, comp.data_ptr(), comp.numel(), bits, out.data_ptr(), n)
    assert res["n_symbols"] == n
    assert hb.gen_verify_device(c, m, SEED, 0, n, out.data_ptr()) == 0
    # oracle on the first 2^22 symbols
    k = 1 << 22
    kb = hb.gen_count_bits_device(c, m, SEED, 0, k)
    host = comp[: (kb + 7) // 8 + 16].cpu().numpy()
    st = O.Stream(m.tree, np.concatenate([host, np.zeros(16, np.uint8)]), kb, k)
    assert np.array_equal(O.simple_decode(st), out[:k].cpu().numpy())
    cb.close()
    c.close()
    del comp, out
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("wpt", [4, 8, 16])
@pytest.mark.parametrize("name", ["paper1", "world192", "kjv", "bible", "english4m", "dna4m", "fib1m", "uniform1m"])
def test_sync_paths_agree(dev, name, wpt):
    """The transducer sync kernel (default on full tiles) and the probe sync kernel
    must give the same bytes, symbol count and shard map."""
    f = _stream(name)
    outs = []
    for path in ("fsm", "probe", "auto", "fsm:2", "fsm:1"):
        c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream, words_per_thread=wpt)
        if ":" in path:      # transducer table in 4 / 2 copies on disjoint banks (8-word subsequences)
            c.set_sync_copies(int(path.split(":")[1]))
        c.set_sync_path(path.split(":")[0])
        cb = hb.Codebook(c, f.tree)
        got, res, _ = _decode_dev(c, cb, f, dev)
        comp = _to_dev(f.data, f.nbytes, dev)
        d_map = torch.zeros(32, dtype=torch.int64, device=dev)
        hb.shard_map(c, cb, comp.data_ptr(), comp.numel(), f.bits, f.bits, d_map.data_ptr())
        c.sync()
        outs.append((got, res["n_symbols"], res["launches"], d_map.cpu().numpy().copy()))
        cb.close()
        c.close()
    assert O.sha256(outs[0][0]) == O.digest(name)
    for k in (1, 2, 3, 4):
        assert outs[0][1] == outs[k][1] == f.usize
        assert np.array_equal(outs[0][0], outs[k][0])
        assert np.array_equal(outs[0][3], outs[k][3])
    assert outs[0][2] >= outs[1][2]   # the transducer path adds a launch when a partial tile remains


@pytest.mark.gpu
@pytest.mark.parametrize("wpt", [4, 8])
@pytest.mark.parametrize("lengths", [[2, 2, 2, 4, 4, 4, 4], [7] * 64 + [8] * 128,
                                     [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 12], [3] * 8,
                                     list(range(1, 31)) + [30],
                                     [2] + [3] * 5 + list(range(4, 33)) + [32]])
def test_hard_codes(dev, lengths, wpt):
    """chains that merge late or never; codewords of up to 32 bits (marker entries, three
    table levels) -- symbols drawn uniformly so that the long ones occur"""
    ctx = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream, words_per_thread=wpt)
    tree, codes = O.tree_from_lengths(lengths)
    rng = np.random.default_rng(len(lengths))
    syms = rng.integers(0, len(lengths), 1 << 20).astype(np.uint8)
    data, bits = O.encode_with_codes(codes, syms)
    f = hb.HuffFile(tree, data, bits, syms.size)
    cb = hb.Codebook(ctx, tree)
    got, res, _ = _decode_dev(ctx, cb, f, dev)
    assert res["n_symbols"] == syms.size and np.array_equal(got, syms)
    cb.close()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("wpt", [4, 8, 16])
@pytest.mark.parametrize("name", ["paper1", "world192", "kjv", "ecoli", "english4m", "dna4m", "fib1m", "uniform1m"])
def test_emit_paths_agree(dev, name, wpt):
    """word-granular staging stores (E64-table, default where the code length allows) and
    byte stores (E-table) give the same bytes, at every output alignment"""
    f = _stream(name)
    for path in ("words", "bytes", "auto", "flat", "words32", "words32:11:3", "words32:9:1", "words32:14:0", "words32:13:1", "words32:15:0", "words32w", "words32w:12:0", "words32w:15:0", "words32w1", "words32w1:14:0",
                 "words64w", "words64w:11:2", "words64w:12:0", "words64w:9:3"):
        c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream, words_per_thread=wpt)
        if ":" in path:     # E32-table geometry: index bits, log2(copies)
            _, wf, rs = path.split(":")
            c.set_emit_table(int(wf), int(rs))
        name0 = path.split(":")[0]
        if name0 == "words32w1":          # one subsequence per lane instead of two
            c.set_emit_lane_subsequences(1)
            name0 = "words32w"
        c.set_emit_path(name0)
        cb = hb.Codebook(c, f.tree)
        for off in (0, 1, 2, 3, 7):
            got, res, raw = _decode_dev(c, cb, f, dev, out_offset=off)
            assert res["n_symbols"] == f.usize and O.sha256(got) == O.digest(name), (path, off)
            assert not raw[off + f.usize:].any() and not raw[:off].any()
        cb.close()
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hello", "paper1", "world192", "ecoli", "fib", "english", "dna", "uniform8"])
def test_device_built_tables_match_host_construction(ctx, name):
    """hb_build_tables_kernel (one thread per table entry, walking the uploaded node array)
    against csrc/hb_lut.c's host construction, entry by entry"""
    models = {"fib": hb.MODEL_FIBONACCI, "english": hb.MODEL_ENGLISH, "dna": hb.MODEL_DNA, "uniform8": hb.MODEL_UNIFORM8}
    if name in models:
        tree = hb.Model(models[name]).tree
    else:
        tree = _stream(name).tree
    lut = hb.build_lut(tree)
    cb = hb.Codebook(ctx, tree)
    assert np.array_equal(cb.table("lut"), lut["entries"])
    for key in ("stab", "etab", "e64"):
        assert np.array_equal(cb.table(key), lut[key]), key
    fsm = cb.table("fsm")
    assert fsm.size == lut["fsm_states"] * 256
    if fsm.size:
        assert np.array_equal(fsm, lut["fsm"])
    cb.close()


@pytest.mark.gpu
def test_tree_with_more_than_256_internal_nodes(ctx, dev):
    """no transducer table: the probe sync kernel does every tile (dispatch in launch_map)"""
    lengths = [8] * 212 + [9] * 88
    tree, codes = O.tree_from_lengths(lengths)
    rng = np.random.default_rng(3)
    syms = rng.integers(0, 300, 1 << 20)
    data, bits = O.encode_with_codes(codes, syms)
    f = hb.HuffFile(tree, data, bits, syms.size)
    cb = hb.Codebook(ctx, tree)
    assert cb.table("fsm").size == 0
    got, res, _ = _decode_dev(ctx, cb, f, dev)
    assert res["n_symbols"] == syms.size and np.array_equal(got, (syms & 255).astype(np.uint8))
    cb.close()


@pytest.mark.gpu
@pytest.mark.parametrize("geom", [(0, -1), (8, 4), (10, 4), (11, 3), (12, 2), (12, 0), (9, 1)])
@pytest.mark.parametrize("name", ["paper1", "world192", "kjv", "ecoli", "bible", "english4m", "dna4m", "fib1m", "uniform1m"])
def test_flat_emit_table_geometries(dev, name, geom):
    """hb_emitf_kernel with every EP-table shape (index bits, log2 copies): same bytes, at
    several output alignments; nothing written outside the slice"""
    f = _stream(name)
    c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream)
    c.set_emit_path("flat")
    c.set_emit_table(*geom)
    cb = hb.Codebook(c, f.tree)
    for off in (0, 1, 6, 11):
        got, res, raw = _decode_dev(c, cb, f, dev, out_offset=off)
        assert res["n_symbols"] == f.usize and O.sha256(got) == O.digest(name), (geom, off)
        assert not raw[off + f.usize:].any() and not raw[:off].any()
    cb.close()
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("lengths", [[2, 2, 2, 4, 4, 4, 4], [4] * 15 + [8] * 16, [3] * 7 + [6] * 8, [6] * 63 + [12] * 64],
                         ids=["even", "mult4", "mult3", "mult6"])
def test_common_length_factor_is_no_cliff(dev, lengths):
    """Round 1 decoded a code whose lengths are all even 18 times slower than English text of
    the same size (entry offsets off the residue class of the codeword starts never merge with
    the true chain and were followed through whole tiles).  Such offsets cannot occur
    (hb_stream_args.gmod) and are skipped now: the decode must be byte-exact AND within a
    factor of two of the English stream's time -- on one GPU and sharded over all of them."""
    rng = np.random.default_rng(5)
    n = 1 << 24
    c = hb.Context(0, stream=torch.cuda.current_stream().cuda_stream)

    def best_ms(tree, data, bits, syms):
        cb = hb.Codebook(c, tree)
        nb = (bits + 7) // 8
        comp = torch.zeros((nb + 15) // 16 * 16 + 32, dtype=torch.uint8, device=dev)
        comp[:nb] = torch.from_numpy(np.ascontiguousarray(data[:nb])).to(dev)
        out = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
        best = None
        for _ in range(5):
            res = hb.decode_device(c, cb, comp.data_ptr(), comp.numel(), bits, out.data_ptr(), n)
            best = res["ms_total"] if best is None else min(best, res["ms_total"])
        assert res["n_symbols"] == n and np.array_equal(out[:n].cpu().numpy(), syms)
        cb.close()
        return best

    p = np.array([2.0 ** -l for l in lengths])
    syms = rng.choice(len(lengths), size=n, p=p / p.sum()).astype(np.uint8)
    tree, codes = O.tree_from_lengths(lengths)
    data, bits = O.encode_with_codes(codes, syms)
    t_code = best_ms(tree, data, bits, syms)
    m = hb.Model(hb.MODEL_ENGLISH)
    f, esyms = m.huff_file_cpu(7, n)
    t_eng = best_ms(f.tree, f.data, f.bits, esyms)
    c.close()
    # An ODD common factor (3, 6 = 2 * 3 ...): subsequences are 256 bits long, so their starts wander
    # through the residue classes; the probe sync kernel starts every chain at the first offset of the
    # right class (hb_first_entry) -- slower than the transducer kernel, but no cliff (round 2: 35x).
    fast = all(l % 3 for l in lengths)
    assert t_code < (2.0 if fast else 4.0) * t_eng, (t_code, t_eng)
    # sharded: every shard knows where it begins in the stream (hb_multi sets the origin)
    mm = hb.Multi(0)
    mm.load(tree, data, bits)
    best = min(mm.decode()["ms_device_max"] for _ in range(4))
    out = np.zeros(n, dtype=np.uint8)
    mm.download(out)
    mm.close()
    assert np.array_equal(out, syms)
    assert best < (2.0 if fast else 4.0) * t_eng, (best, t_eng)
