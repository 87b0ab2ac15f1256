#!/usr/bin/env python
"""bench.py -- headline measurement of the B200 speculative parallel Huffman decoder.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): decoded GB/s, device-timed, on the synthetic English-like
stream of config 4 (2^30 symbols per GPU, order-0 histogram of bible.txt, encoded
in the reference's .huff bit format by the bundled generator).  A step is one
whole decode of the stream(s): N=1 decodes the 2^30-symbol stream; N>1 decodes
one stream of N * 2^30 symbols partitioned by compressed byte range, one shard
per GPU, with one NCCL all-gather of the 32-entry boundary maps (weak scaling).
Prints ONE JSON line on rank 0.  Besides the headline the line carries, under
"secondary", the same measurement (fewer steps, byte-verified) of BASELINE config 5
at its stated size (fib16g: ONE 2^34-symbol stream, whole on one GPU, split over
N), of fib4g, and of english1g under strong scaling (2^30 symbols split over N).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

SEED = 0x48554646  # "HUFF"
TIMING_RING = 4096   # most steps hb_ctx_timing_begin keeps per-kernel events for
DUMP_SAMPLE = 1 << 21    # decoded bytes sampled by --dump-outputs (fixed positions, SEED)
DUMP_BLOCK = 1 << 20     # --dump-outputs sums the decoded bytes per block of this many
PEER = {"on": False, "seq": 0}   # map exchange by peer stores (hb_shard_exchange); seq advances on every rank alike
WORKLOADS = {
    # name: (model kind, log2 symbols, default scaling, description).  weak: that many symbols
    # per GPU of one N-times-larger stream; strong: that many symbols in total, split over N
    "english1g": (0, 30, "weak", "synthetic English-like (order-0 histogram of bible.txt), 2^30 symbols"),
    "fib4g": (1, 32, "weak", "synthetic Fibonacci-skewed 256-symbol alphabet (max code length 24), 2^32 symbols"),
    "fib16g": (1, 34, "strong", "BASELINE config 5 at its stated size: ONE Fibonacci-skewed stream of 2^34 symbols "
                                "(max code length 24), whole on one GPU or split over N"),
    "english64m": (0, 26, "weak", "synthetic English-like, 2^26 symbols (quick check)"),
}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML (the interface behind
    nvidia-smi's clocks.sm / clocks_event_reasons.*) every ~10 ms by a thread;
    only samples taken inside the timed region are kept."""

    def __init__(self, index):
        self.index = index
        self.samples = []   # (t, sm_mhz, reasons_bitmask)
        self.stop_flag = False
        self.ok = False
        self.sm_max = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            # NVML indexes physical devices; map through CUDA_VISIBLE_DEVICES when it is numeric
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def start(self):
        if not self.ok:
            return
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.th.join(timeout=2)
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        sm = sorted(s[1] for s in inside)
        mask = 0
        for s in inside:
            mask |= s[2]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max,
                "samples": len(inside), "reasons": sorted(v for k, v in names.items() if mask & k)}


# ---------------------------------------------------------------------------------
# CPU legs (the oracle / the compiled reference are used ONLY here, as the baseline)
# ---------------------------------------------------------------------------------

def cpu_sample(kind, log2n):
    """First 2^log2n symbols of the workload, built by the CPU generator."""
    import numpy as np
    import huffmandecoderongpus_b200 as hb
    import oracle_lib as O
    m = hb.Model(kind)
    f, syms = m.huff_file_cpu(SEED, 1 << log2n)
    return O.Stream(f.tree, f.data, f.bits, f.usize), syms


def cpu_time_paths(st, syms, reps):
    """Reference protocol (framework/decodeUtil.c:30-70): first run byte-checked,
    min wall time over the runs.  Returns {path: seconds}, kind."""
    import numpy as np
    import oracle_lib as O
    use_ref = O.ref() is not None and st.bits < 2 ** 31
    out = {}

    def timed(fn):
        best = None
        for r in range(reps):
            t0 = time.perf_counter()
            got = fn()
            dt = time.perf_counter() - t0
            if r == 0:
                assert np.array_equal(got, syms), "CPU baseline output differs from the generated symbols"
            best = dt if best is None else min(best, dt)
        return best

    if use_ref:
        out["simpleDecode"] = timed(lambda: O.ref_decode(st, "simpleDecode"))
        out["jumptableApproach_jb8"] = timed(lambda: O.ref_decode(st, "jumptableApproach", 8))
        kind = "reference"
    else:
        out["simpleDecode"] = timed(lambda: O.simple_decode(st))
        out["jumptableApproach_jb8"] = timed(lambda: O.jumptable_decode(st, 8))
        kind = "port"
    return out, kind


def run_reference_arm(args, kind, desc, scaling="weak"):
    """--impl reference: the reference's own CPU decode path on this box's host
    cores (single-threaded: the reference has no threads), each step a bounded
    sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    log2s = min(args.cpu_sample_log2, 26)
    st, syms = cpu_sample(kind, log2s)
    import oracle_lib as O
    use_ref = O.ref() is not None
    fn = (lambda: O.ref_decode(st, "jumptableApproach", 8)) if use_ref else (lambda: O.jumptable_decode(st, 8))
    import numpy as np
    for _ in range(max(args.warmup, 1)):
        got = fn()
    assert np.array_equal(got, syms)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    dt = time.perf_counter() - t0
    gbs = args.steps * syms.size / dt / 1e9
    sample = (f"first 2^{log2s} symbols of the workload ({st.nbytes} compressed bytes), "
              f"{'unmodified reference' if use_ref else 'oracle port of'} jumptableApproach(jumpbits=8), 1 thread")
    line = {
        "impl": "reference", "metric": "decoded_GB_per_s", "value": gbs, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": args.workload, "description": desc, "sample": sample},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": 1,
                         "kind": "reference" if use_ref else "port", "sample": sample},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------

class Job:
    """One workload on this rank: the stream built on the device (setup), cut into byte-range
    shards, decoded through the C ABI; verified against regenerated symbols."""

    def __init__(self, args, ctx, name, scaling, world, rank, dev):
        import numpy as np
        import torch
        import torch.distributed as dist
        import huffmandecoderongpus_b200 as hb
        self.hb, self.torch, self.dist, self.np = hb, torch, dist, np
        self.args, self.ctx, self.world, self.rank, self.dev = args, ctx, world, rank, dev
        kind, log2n, dflt, self.desc = WORKLOADS[name]
        self.name, self.kind = name, kind
        self.scaling = dflt if scaling == "auto" else scaling
        self.n_total = (1 << log2n) * (world if self.scaling == "weak" else 1)
        self.model = hb.Model(kind)
        self.cb = hb.Codebook(ctx, self.model.tree)
        # ---- build the stream on the device (setup, untimed) ----
        self.bits_total = hb.gen_count_bits_device(ctx, self.model, SEED, 0, self.n_total)
        self.nbytes_total = (self.bits_total + 7) // 8
        per = (self.nbytes_total // world) // 16 * 16
        a = rank * per
        b = self.nbytes_total if rank == world - 1 else (rank + 1) * per
        last = rank == world - 1
        whole = torch.zeros((self.nbytes_total + 15) // 16 * 16 + 64, dtype=torch.uint8, device=dev)
        assert hb.gen_encode_device(ctx, self.model, SEED, 0, self.n_total, whole.data_ptr(), whole.numel()) == self.bits_total
        halo_end = min(self.nbytes_total, b + 16)
        self.halo_bytes = halo_end - a
        self.comp = torch.zeros((halo_end - a + 15) // 16 * 16 + 16, dtype=torch.uint8, device=dev)
        self.comp[: halo_end - a] = whole[a:halo_end]
        del whole
        torch.cuda.empty_cache()
        ctx.set_shard_origin(a)    # this rank's shard begins at byte a of the stream
        self.bits_own = self.bits_total - 8 * a if last else 8 * (b - a)
        self.bits_avail = self.bits_own if last else min(self.bits_total - 8 * a, 8 * (halo_end - a))
        self.comp_bytes_own = (self.bits_own + 7) // 8
        n_share = self.n_total // world
        self.cap = int(n_share * 1.02) + (1 << 16)
        self.out = torch.zeros(self.cap + 64, dtype=torch.uint8, device=dev)
        self.my_map = torch.zeros(32, dtype=torch.int64, device=dev)
        self.all_maps = torch.zeros(32 * world, dtype=torch.int64, device=dev)
        self.eb = torch.zeros(4, dtype=torch.int64, device=dev)
        # ---- correctness of this very configuration (untimed) ----
        self.barrier()             # ranks aligned: hb_shard_exchange gives a left neighbour 5 s to deliver its map
        res = self.step(want_result=True)
        self.n_mine, self.out_base = res["n_symbols"], res["out_base"]
        self.launches_per_step = res["launches"] + (1 if world > 1 else 0)   # + hb_exchange_kernel / hb_compose_kernel
        self.verify_device(self.out, "device-resident decode")

    def verify_device(self, out_tensor, what):
        hb, torch, dist = self.hb, self.torch, self.dist
        bad = hb.gen_verify_device(self.ctx, self.model, SEED, self.out_base, self.n_mine, out_tensor.data_ptr())
        tot = torch.tensor([self.n_mine, bad], dtype=torch.int64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(tot)
        assert int(tot[0]) == self.n_total and int(tot[1]) == 0, \
            f"{self.name}: {what} mismatch: {tot.tolist()} vs {self.n_total} symbols"

    def dump_outputs(self, out_dir):
        """What the last step left for its caller, as DIR/<name>.npy (float32 / float64, about 25 MB):
        n_symbols [symbols decoded, output base in the stream], decoded_sample (bytes at DUMP_SAMPLE
        positions drawn with SEED, positions in decoded_sample_index) and decoded_block_sums (sum of
        every DUMP_BLOCK bytes, so that a difference anywhere in the output shows).  The symbol count
        is the verified first step's: every step decodes the same stream.  Ranks > 1 add _rank<r>."""
        np, torch = self.np, self.torch
        n = int(self.n_mine)
        out = self.out[:n]
        idx = np.sort(np.random.default_rng(SEED).integers(0, n, size=min(n, DUMP_SAMPLE)))
        whole = n // DUMP_BLOCK * DUMP_BLOCK
        sums = out[:whole].view(-1, DUMP_BLOCK).sum(dim=1, dtype=torch.int64)
        if whole < n:
            sums = torch.cat([sums, out[whole:].sum(dtype=torch.int64).view(1)])
        arrays = {
            "n_symbols": np.array([n, self.out_base], dtype=np.float64),
            "decoded_sample": out[torch.from_numpy(idx).to(self.dev)].cpu().numpy().astype(np.float32),
            "decoded_sample_index": idx.astype(np.float64),
            "decoded_block_sums": sums.cpu().numpy().astype(np.float64),
        }
        os.makedirs(out_dir, exist_ok=True)
        suffix = f"_rank{self.rank}" if self.world > 1 else ""
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + suffix + ".npy"), a)

    def step(self, want_result=False):
        hb, c = self.hb, self.comp
        if self.world == 1:    # one GPU, one shard: the single-GPU entry point
            return hb.decode_device(self.ctx, self.cb, c.data_ptr(), c.numel(), self.bits_own,
                                    self.out.data_ptr(), self.cap, want_result=want_result)
        hb.shard_map(self.ctx, self.cb, c.data_ptr(), c.numel(), self.bits_own, self.bits_avail, self.my_map.data_ptr())
        if self.world > 1:
            self.exchange()
            ebp = self.eb.data_ptr()
        else:
            ebp = None
        return hb.shard_emit(self.ctx, self.cb, c.data_ptr(), c.numel(), self.bits_own, self.bits_avail, ebp,
                             self.out.data_ptr(), self.cap, want_result=want_result)

    def exchange(self):
        """shard maps -> this rank's (entry offset, output base): ONE kernel of peer stores over NVLink
        (hb_shard_exchange) or, with --exchange nccl, NCCL's all-gather + hb_shard_compose"""
        if PEER["on"]:
            PEER["seq"] += 1
            self.hb.shard_exchange(self.ctx, PEER["seq"], self.eb.data_ptr())
        else:
            self.dist.all_gather_into_tensor(self.all_maps, self.my_map)
            self.hb.shard_compose(self.ctx, self.all_maps.data_ptr(), self.world, self.rank, self.eb.data_ptr())

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, steps, warmup, sampler=None):
        """W untimed steps, then exactly K steps between barrier + synchronize on both sides,
        CUDA events on the launching stream, max over ranks."""
        torch = self.torch
        for _ in range(max(warmup - 1, 0)):
            self.step()
        self.barrier()
        if sampler is not None:
            sampler.start()
        self.ctx.timing_begin(min(steps, TIMING_RING))   # per-kernel split over the first TIMING_RING steps
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        self.barrier()
        w0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            self.step()
        e1.record()
        self.barrier()
        w1 = time.perf_counter()
        ms = e0.elapsed_time(e1)
        phases = self.ctx.timing_collect()
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        ms_step = float(t[0]) / steps
        return ms_step, phases, (w0, w1)

    def summary(self, ms_step, phases):
        peak, _ = measured_peak()
        b_alg = self.comp_bytes_own + self.n_mine
        k_total = phases["total"] / max(phases["steps"], 1)
        return {"value": self.n_total / (ms_step * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_step,
                "scaling": self.scaling, "symbols_total": self.n_total,
                "compressed_bytes_total": int(self.nbytes_total), "max_code_length": self.model.maxlen,
                "compressed_input_GB_per_s": self.nbytes_total / (ms_step * 1e-3) / 1e9,
                "decode_frac_rank0": b_alg / (k_total * 1e-3) / 1e9 / peak,
                "kernel_ms_rank0": {k: phases[k] / max(phases["steps"], 1) for k in ("sync", "scan", "emit")},
                "verified": "every output byte against regenerated symbols, on the device"}

    def close(self):
        self.cb.close()
        del self.comp, self.out
        self.torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="english1g", choices=list(WORKLOADS))
    ap.add_argument("--scaling", default="auto", choices=["auto", "weak", "strong"],
                    help="weak: the workload's symbols per GPU; strong: in total (auto: the workload's default)")
    ap.add_argument("--wpt", type=int, default=0, help="words per thread (0 = library default)")
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--ep-wf", type=int, default=0, help="EP-table index bits of the flat emit kernel (0 = auto)")
    ap.add_argument("--ep-copies-log2", type=int, default=-1, help="log2 of the EP-table copies (-1 = auto)")
    ap.add_argument("--emit-path", default="auto", choices=["auto", "bytes", "words", "flat", "words32", "words32w", "words64w"],
                    help="emit kernel A/B (auto = words)")
    ap.add_argument("--emit-spl", type=int, default=1, choices=[1, 2], help="subsequences per lane of the warp-autonomous emit kernel")
    ap.add_argument("--sync-copies-log2", type=int, default=-1, help="transducer table copies in the sync kernel (log2; -1 = auto)")
    ap.add_argument("--sync-path", default="auto", choices=["auto", "probe", "fsm"],
                    help="sync kernel A/B")
    ap.add_argument("--cpu-sample-log2", type=int, default=27)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--host-chunk-mib", type=int, default=0,
                    help="chunk size of the pipelined host path (0 = library default)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the 32-entry shard maps travel -- one kernel of peer stores over NVLink "
                         "(hb_shard_exchange) or NCCL all-gather + hb_shard_compose")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one decoded as DIR/<name>.npy "
                         "(a fixed sample, block sums and the symbol count) to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path decoded")
    if args.warmup < 3:
        args.warmup = 3   # timing rule: at least three warm-up steps
    kind, log2n, dflt_scaling, desc = WORKLOADS[args.workload]
    scaling = dflt_scaling if args.scaling == "auto" else args.scaling

    if args.impl == "reference":
        run_reference_arm(args, kind, desc, scaling)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import huffmandecoderongpus_b200 as hb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            sys.exit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ctx = hb.Context(local, stream=torch.cuda.current_stream().cuda_stream,
                     words_per_thread=args.wpt, ctas_per_sm=args.ctas_per_sm)
    ctx.set_sync_path(args.sync_path)
    ctx.set_sync_copies(args.sync_copies_log2)
    ctx.set_emit_lane_subsequences(args.emit_spl)
    if args.host_chunk_mib:
        ctx.set_host_chunk(args.host_chunk_mib << 20)
    ctx.set_emit_path(args.emit_path)
    ctx.set_emit_table(args.ep_wf, args.ep_copies_log2)
    if world > 1 and args.exchange == "peer":
        # exchange tables: one 64-byte IPC handle per rank, passed around once; all ranks or none
        ok = 1
        try:
            handles = [None] * world
            dist.all_gather_object(handles, hb.peer_export(ctx))
            hb.peer_connect(ctx, rank, handles)
        except Exception as e:                      # no IPC / no peer access on this box: NCCL
            print(f"rank {rank}: peer exchange unavailable ({e}); using NCCL", file=sys.stderr)
            ok = 0
        t = torch.tensor([ok], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        dist.barrier()
        PEER["on"] = bool(int(t[0]))

    job = Job(args, ctx, args.workload, scaling, world, rank, dev)
    model, n_total, n_mine = job.model, job.n_total, job.n_mine

    # ---- timed region ---------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    ms_step, phases, (w0, w1) = job.timed(args.steps, args.warmup, sampler)
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    if args.dump_outputs:
        job.dump_outputs(args.dump_outputs)     # before the e2e leg reuses job.out
    value = n_total / (ms_step * 1e-3) / 1e9
    in_gbs = job.nbytes_total / (ms_step * 1e-3) / 1e9

    # ---- roofline of the dominant kernel (rank 0's CUDA events over the timed steps) --
    peak, peak_src = measured_peak()
    b_alg = job.comp_bytes_own + n_mine             # SURVEY 8(d): compressed read once + decoded written once
    k_ms = {k: phases[k] / max(phases["steps"], 1) for k in ("sync", "scan", "emit", "total")}
    dom = max(("sync", "emit"), key=lambda k: k_ms[k])
    sync_name = "hb_sync_kernel" if args.sync_path == "probe" else "hb_fsm_sync_kernel"
    emit_name = ctx.last_emit_kernel() or "hb_emit_kernel"
    dom_name = {"sync": sync_name, "emit": emit_name}[dom]
    achieved = b_alg / (k_ms[dom] * 1e-3) / 1e9
    # DRAM bytes per launch of that kernel from the committed ncu --set full capture of this
    # same command (profiles/traffic.json); only quoted for the configuration it was taken on
    traffic = None
    try:
        if args.workload == "english1g" and (args.wpt or 8) == 8 and world == 1 and scaling == "weak":
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f)["kernels"][dom_name]["dram_bytes"]
    except Exception:
        traffic = None
    roofline = {
        "bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": b_alg,
        "kernel_ms": {sync_name: k_ms["sync"], "hb_scan_*+hb_fix": k_ms["scan"], emit_name: k_ms["emit"]},
        "decode_achieved": b_alg / (k_ms["total"] * 1e-3) / 1e9,
        "decode_frac": b_alg / (k_ms["total"] * 1e-3) / 1e9 / peak,
        "kernel_share_of_step": k_ms[dom] / k_ms["total"],
    }

    # ---- end to end through host buffers: the library's own host-buffer entry points --
    e2e = None
    if not args.no_e2e:
        h_comp = torch.empty(job.comp.numel(), dtype=torch.uint8, pin_memory=True)
        h_comp.copy_(job.comp)
        h_out = torch.empty(job.cap + 64, dtype=torch.uint8, pin_memory=True)
        torch.cuda.synchronize()
        steps_e = max(args.e2e_steps, 1)
        hc, ho = h_comp.numpy(), h_out.numpy()[: job.cap]

        def e2e_step():
            if world == 1:
                # the user-facing call: host buffers in, host buffer out (chunked, overlapped)
                return hb.decode_host(ctx, model.tree, hc, job.bits_total, ho)
            # one process per GPU: upload + map | all-gather of the maps | compose, emit + download
            hb.shard_map_host(ctx, job.cb, hc, job.halo_bytes, job.bits_own, job.bits_avail, job.my_map.data_ptr())
            job.exchange()
            return hb.shard_emit_host(ctx, job.cb, job.eb.data_ptr(), ho)

        r = e2e_step()
        job.barrier()
        t0 = time.perf_counter()
        for _ in range(steps_e):
            r = e2e_step()
        job.barrier()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t[0])
        # the WHOLE host-side result, every rank: back to the device, against regenerated symbols
        assert r["n_symbols"] == n_mine, (r["n_symbols"], n_mine)
        job.out.zero_()
        job.out[:n_mine].copy_(h_out[:n_mine])
        job.verify_device(job.out, "end-to-end (host buffers) decode")
        e2e = {"value": n_total * steps_e / dt / 1e9, "unit": "GB/s",
               "h2d_bytes_per_step": int(job.comp_bytes_own), "d2h_bytes_per_step": int(n_mine),
               "steps": steps_e, "ms_per_step": dt / steps_e * 1e3,
               "verified": "all output bytes of every rank",
               "path": "hb_decode_host (pinned host buffers, chunked upload/decode/download overlap)" if world == 1
                       else "per rank: hb_shard_map_host (pinned H2D + map) | " +
                            ("hb_shard_exchange (peer stores) | " if PEER["on"] else "all_gather of 32-entry maps + hb_shard_compose | ") +
                            "hb_shard_emit_host (emit + pinned D2H)"}
        del h_comp, h_out, hc, ho

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only) ----------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        log2s = min(args.cpu_sample_log2, log2n)
        st, syms = cpu_sample(kind, log2s)
        secs, ckind = cpu_time_paths(st, syms, reps=3)
        best = min(secs, key=secs.get)
        cpu = {"value": syms.size / secs[best] / 1e9, "unit": "GB/s", "cores": 1, "kind": ckind,
               "path": best,
               "sample": f"first 2^{log2s} symbols of the workload ({st.nbytes} compressed bytes), "
                         f"min of 3 runs, first run byte-checked, 1 thread of {os.cpu_count()} host CPUs",
               "all_paths_GBps": {k: syms.size / v / 1e9 for k, v in secs.items()}}

    head = {"symbols_total": n_total, "compressed_bytes_total": int(job.nbytes_total),
            "bits_total": int(job.bits_total), "max_code_length": model.maxlen,
            "launches_per_step": job.launches_per_step}
    job.close()

    # ---- secondary workloads: same measurement, fewer steps, byte-verified -----------------
    secondary = {}
    if not args.no_secondary and args.workload == "english1g" and scaling == "weak":
        plan = [("fib4g", "weak", 10), ("fib16g", "strong", 5)]
        if world > 1:
            plan.append(("english1g", "strong", 30))
        for name, sc, k in plan:
            try:
                j = Job(args, ctx, name, sc, world, rank, dev)
                ms2, ph2, _ = j.timed(k, 3)
                key = name if sc == WORKLOADS[name][2] else f"{name}_{sc}"
                secondary[key] = dict(j.summary(ms2, ph2), steps=k, warmup=3)
                j.close()
            except torch.cuda.OutOfMemoryError as e:   # pragma: no cover
                secondary[name] = {"skipped": "out of device memory: " + str(e)[:80]}
                torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": "decoded_GB_per_s", "value": value, "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": args.workload, "description": desc + (" per GPU" if scaling == "weak" else " in total"),
                       "seed": SEED,
                       "symbols_total": head["symbols_total"], "compressed_bytes_total": head["compressed_bytes_total"],
                       "bits_total": head["bits_total"], "max_code_length": head["max_code_length"],
                       "words_per_thread": args.wpt or 8, "sync_path": args.sync_path, "emit_path": args.emit_path,
                       "parallelism": (f"byte-range shards x{world}, maps exchanged by one kernel of peer stores over NVLink (hb_shard_exchange)"
                                       if PEER["on"] else f"byte-range shards x{world}, 1 NCCL all-gather of 32-entry maps") if world > 1 else "single GPU",
                       "l2": "inputs and outputs larger than L2 (no flush needed)",
                       "compressed_input_GB_per_s": in_gbs},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": head["launches_per_step"] * args.steps,
            "clocks": clocks,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if PEER["on"]:          # unmap the neighbours' exchange tables everywhere before any of them is freed
        hb.peer_disconnect(ctx)
        dist.barrier()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
