"""One process, N devices (hb_multi_*, b200ApproachMulti): byte-range shards, maps exchanged
by peer stores (hb_shard_exchange), and the exchange kernel itself over contexts of this process.  Runs with however many GPUs the box has (1 works: a single shard); on a
multi-GPU box the 2-, 4- and 8-device splits are exercised as well."""
import numpy as np
import pytest

import oracle_lib as O
import huffmandecoderongpus_b200 as hb

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SEED = 0x48554646


def _counts():
    n = torch.cuda.device_count()
    return [k for k in (1, 2, 3, 4, 8) if k <= n]


def _stream(name):
    if name in O.STANDINS:
        return O.standin(name)[0]
    p = O.corpus_path(name)
    if p is None:
        pytest.skip(f"{name} corpus not present")
    return hb.HuffFile.load(p)


@pytest.mark.parametrize("name", ["hello", "paper1", "world192", "kjv", "ecoli", "bible", "english4m", "dna4m", "fib1m", "uniform1m"])
def test_multi_host_buffers(name):
    """hb_multi_decode_host: upload, shard maps, peer exchange, compose, emit, download"""
    f = _stream(name)
    for n in _counts():
        m = hb.Multi(n)
        out = np.zeros(f.usize + 16, dtype=np.uint8)
        res = m.decode_host(f.tree, f.data, f.bits, out[: f.usize])
        assert res["n_symbols"] == f.usize, (n, res)
        assert O.sha256(out[: f.usize]) == O.digest(name), n
        assert not out[f.usize:].any()
        assert sum(res["shard_symbols"]) == f.usize
        # a second call on the same object (cached code tables and buffers)
        out[:] = 0
        res = m.decode_host(f.tree, f.data, f.bits, out[: f.usize])
        assert O.sha256(out[: f.usize]) == O.digest(name), n
        m.close()


def test_multi_output_too_small():
    f = _stream("paper1")
    m = hb.Multi(_counts()[-1])
    out = np.zeros(f.usize - 5, dtype=np.uint8)
    with pytest.raises(hb.HuffError) as e:
        m.decode_host(f.tree, f.data, f.bits, out)
    assert e.value.code == -6
    m.close()


@pytest.mark.parametrize("kind,log2n", [(0, 24), (1, 25), (2, 22)])
def test_multi_resident_generate_decode_verify(kind, log2n):
    """one synthetic stream built on the devices, decoded resident, every slice verified"""
    for n in _counts():
        m = hb.Multi(n)
        bits = m.generate(kind, SEED, 1 << log2n)
        assert bits > 0
        for _ in range(2):
            res = m.decode()
            assert res["n_symbols"] == 1 << log2n, (n, res)
        assert m.verify(kind, SEED) == 0
        # and the bytes themselves against the CPU generator
        out = np.zeros(1 << log2n, dtype=np.uint8)
        m.download(out)
        want = hb.Model(kind).symbols_cpu(SEED, 0, 1 << log2n)
        assert np.array_equal(out, want), n
        m.close()


def test_multi_load_truncated_stream():
    """a stream cut inside a codeword: the cut-off codeword emits nothing, on any split"""
    f = _stream("paper1")
    st = O.load_huff(O.corpus_path("paper1"))
    for bits in (f.bits - 1, f.bits - 7, 100001):
        want = O.simple_decode(st, bits=bits)
        for n in _counts():
            m = hb.Multi(n)
            out = np.zeros(want.size + 8, dtype=np.uint8)
            res = m.decode_host(f.tree, f.data, bits, out[: want.size])
            assert res["n_symbols"] == want.size, (bits, n)
            assert np.array_equal(out[: want.size], want)
            m.close()


def test_onethread_matches_oracle():
    """the reference's onethread debug approach (framework/onethread.cu:13-52)"""
    for name in ("hello", "paper1"):
        f = _stream(name)
        ctx = hb.Context(0)
        out = np.zeros(f.usize, dtype=np.uint8)
        res = hb.decode_onethread(ctx, f.tree, f.data, f.bits, out)
        assert res["n_symbols"] == f.usize
        assert O.sha256(out) == O.CORPORA[name][2]
        ctx.close()


@pytest.mark.parametrize("name,nshards,order", [("kjv", 2, "up"), ("kjv", 8, "down"), ("paper1", 3, "down"),
                                                ("ecoli", 4, "down"), ("bible", 5, "up"), ("english4m", 2, "up"),
                                                ("english4m", 8, "down"), ("dna4m", 4, "down"), ("fib1m", 5, "up")])
def test_peer_exchange_replaces_allgather_and_compose(name, nshards, order):
    """hb_shard_exchange: every rank stores its map into the exchange tables of the ranks to its right
    (peer stores) and waits for the maps of the ranks to its left in ONE kernel.  Ranks = contexts of this
    process with their own streams, spread over the devices of the box (one device works: the kernels of
    different streams run side by side); "down" queues the LAST rank first, so that its kernel really has
    to wait for flags that are not there yet.  Three decodes in a row: the ring slots move with seq."""
    f = _stream(name)
    want = O.simple_decode(O.Stream(f.tree, f.data, f.bits, f.usize))
    ndev = torch.cuda.device_count()
    per = (f.nbytes // nshards) // 16 * 16
    bounds = [r * per for r in range(nshards)] + [f.nbytes]
    ctxs = [hb.Context(r % ndev) for r in range(nshards)]
    cbs = [hb.Codebook(c, f.tree) for c in ctxs]
    hb.peer_connect_local(ctxs)
    shards = []
    for r in range(nshards):
        dev = torch.device("cuda", r % ndev)
        a, b = bounds[r], bounds[r + 1]
        last = r == nshards - 1
        bits_own = f.bits - 8 * a if last else 8 * (b - a)
        halo_end = min(f.nbytes, b + 16)
        bits_avail = bits_own if last else min(f.bits - 8 * a, 8 * (halo_end - a))
        nb = halo_end - a
        comp = torch.zeros((nb + 15) // 16 * 16 + 32, dtype=torch.uint8, device=dev)
        comp[:nb] = torch.from_numpy(np.ascontiguousarray(f.data[a:halo_end])).to(dev)
        eb = torch.zeros(4, dtype=torch.int64, device=dev)
        out = torch.zeros(want.size + 64, dtype=torch.uint8, device=dev)
        shards.append((comp, bits_own, bits_avail, eb, out))
    for d in range(ndev):
        torch.cuda.synchronize(d)
    ranks = list(range(nshards)) if order == "up" else list(range(nshards - 1, -1, -1))
    for seq in (1, 2, 3):
        for r in ranks:
            comp, bo, ba, eb, out = shards[r]
            hb.shard_map(ctxs[r], cbs[r], comp.data_ptr(), comp.numel(), bo, ba, 0)
            hb.shard_exchange(ctxs[r], seq, eb.data_ptr())
        pieces, base_expect = [None] * nshards, 0
        results = {}
        for r in ranks:
            comp, bo, ba, eb, out = shards[r]
            results[r] = hb.shard_emit(ctxs[r], cbs[r], comp.data_ptr(), comp.numel(), bo, ba, eb.data_ptr(),
                                       out.data_ptr(), want.size)
        for r in range(nshards):
            res = results[r]
            assert res["out_base"] == base_expect, (seq, r)
            base_expect += res["n_symbols"]
            pieces[r] = shards[r][4][: res["n_symbols"]].cpu().numpy()
            assert int(shards[r][3][2]) == base_expect          # symbols through this rank
        got = np.concatenate(pieces)
        assert got.size == want.size and np.array_equal(got, want), seq
    for cb in cbs:
        cb.close()
    for c in ctxs:
        c.close()


def test_peer_exchange_times_out_instead_of_hanging():
    """a rank whose left neighbour never delivers reports HB_ERR_STATE after the kernel's 5 s limit"""
    f = _stream("paper1")
    ctxs = [hb.Context(0), hb.Context(0)]
    cbs = [hb.Codebook(c, f.tree) for c in ctxs]
    hb.peer_connect_local(ctxs)
    dev = torch.device("cuda", 0)
    nb = f.nbytes
    comp = torch.zeros((nb + 15) // 16 * 16 + 32, dtype=torch.uint8, device=dev)
    comp[:nb] = torch.from_numpy(np.ascontiguousarray(f.data[:nb])).to(dev)
    eb = torch.zeros(4, dtype=torch.int64, device=dev)
    out = torch.zeros(f.usize + 64, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    hb.shard_map(ctxs[1], cbs[1], comp.data_ptr(), comp.numel(), f.bits, f.bits, 0)
    hb.shard_exchange(ctxs[1], 7, eb.data_ptr())          # rank 0 never runs
    with pytest.raises(hb.HuffError) as e:
        hb.shard_emit(ctxs[1], cbs[1], comp.data_ptr(), comp.numel(), f.bits, f.bits, eb.data_ptr(),
                      out.data_ptr(), f.usize)
    assert e.value.code == -9
    for cb in cbs:
        cb.close()
    for c in ctxs:
        c.close()
