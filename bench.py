#!/usr/bin/env python
"""bench.py -- throughput of the BPE-encode hot path (BASELINE.json metric: input GB/s and
Mtokens/s, cl100k_base, 1 GiB synthetic English-like corpus = SURVEY.md 8(d) config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload config2] [--dump-outputs DIR]

A "step" = one pass of the hot path over one batch (the whole workload of this rank).
  value    device-resident: text + doc offsets already in HBM, tokens + offsets left in HBM.  The K steps are
           ENQUEUED back to back on one CUDA stream (b200bpe_encode_device_async: no host synchronisation inside a
           step; the per-step count exchange is an NCCL all-gather enqueued behind the pipeline from a device buffer
           the last kernel fills) and timed with CUDA events recorded on that stream; max over ranks.
  e2e      the same metric through the public host API (Encoding.encode_ordinary_packed ->
           C ABI b200bpe_encode_ordinary_batch) with pinned HOST buffers: H2D of the text, the
           kernels and D2H of tokens + offsets are all inside the timed region.  Its output is compared
           byte for byte with the device-resident result on every rank.
  api      the calls a tiktoken user makes: encode_ordinary_batch(list[str]) (Python marshalling + pageable memory
           through the pinned staging ring) and encode_batch with the default disallowed_special="all" (device scan).
  roofline achieved algorithmic bytes/s of the dominant kernel from CUDA events recorded by the engine around
           that launch, against the measured HBM peak; and the same for the whole pipeline.
  configs  every other BASELINE.json config at its stated size, same method, with a parity flag each.
  strong   ONE 1 GiB corpus split over the ranks (BASELINE asks for "a 1 GB corpus at 1/2/4/8"), next to the weak line.
  cpu_baseline / --impl reference: the reference engine itself (the tiktoken wheel's Rust CoreBPE
           driven through tiktoken.Encoding.encode_ordinary_batch with all host cores) on a bounded
           sample of the same workload; if the wheel cannot be imported, the oracle port.
N > 1 (torchrun, one rank per GPU): documents shard across ranks (weak scaling: every rank has its
own corpus of the configured size); the only exchange is an NCCL all-gather of per-rank counts.
Every rank is gated against the oracle before any number is reported.
--dump-outputs DIR: after the timed steps, rank 0 writes what the last of them left in HBM (see Bench.dump_outputs),
so that two builds run with the same arguments -- hence the same seeded inputs -- can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # the benchmark writes nothing into the source tree (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from tools import corpus  # noqa: E402
import vocab_util as vu   # noqa: E402

WORKLOADS = {
    # name: (encoding, builder, description)
    "config1": ("r50k_base", lambda n, seed: corpus.config1(n, seed), "gpt2/r50k_base, ONE 1 MiB ASCII document (plumbing)"),
    "config2": ("cl100k_base", lambda n, seed: corpus.config2(n, seed), "cl100k_base, english-like, ~64 KiB docs"),
    "config3": ("o200k_base", lambda n, seed: corpus.config3(n, seed), "o200k_base, mixed UTF-8, docs 4-256 KiB"),
    "config4": ("cl100k_base", lambda n, seed: corpus.config4(max(1, round(n / 102.0)), seed), "cl100k_base, ~100 B docs"),
    "config5": ("p50k_base", lambda n, seed: corpus.config5(n, seed), "p50k_base, one code-like document"),
}
DEFAULT_BYTES = {"config1": 1 << 20, "config2": 1 << 30, "config3": 1 << 30, "config4": 1_020_000_000, "config5": 64 << 20}
SEEDS = {"config1": 1001, "config2": 1002, "config3": 1003, "config4": 1004, "config5": 1005}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi DURING the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "10"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None, t_warm=None):
        """Clocks from the samples that arrived inside [t0, t1] (the timed region).  The sampler is started before the
        warm-up steps so that it is already running; when fewer than three samples fall inside the timed region (five
        6.7 ms steps are one or two 10 ms sampling periods) the window is widened to the identical warm-up steps that
        run back to back before it (from t_warm) and the line says so."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        window = "all"
        rows = self.rows
        if t0 is not None:
            rows, window = [r for r in self.rows if t0 <= r[0] <= t1 + 0.02], "timed region"
            if len(rows) < 3 and t_warm is not None:
                rows, window = [r for r in self.rows if t_warm <= r[0] <= t1 + 0.02], "warm-up steps + timed region (back to back)"
        sm, mx, reasons = [], None, set()
        for _, r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


def sample_positions(n: int, k: int, seed: int = 2024) -> np.ndarray:
    """Sorted positions of a fixed, seeded sample of at most k of range(n); all of them when n <= k."""
    if n <= k:
        return np.arange(n, dtype=np.int64)
    return np.unique(np.random.default_rng(seed).integers(0, n, size=k, dtype=np.int64))


def load_reference_engine(pat, ranks, special):
    """The reference engine: installed tiktoken wheel (Rust CoreBPE).  None if not importable."""
    try:
        import tiktoken
        from tiktoken import _tiktoken  # noqa: F401  (make sure it is the native engine)
        return tiktoken.Encoding("bench_ref", pat_str=pat, mergeable_ranks=ranks, special_tokens=special), \
            f"tiktoken=={tiktoken.__version__} wheel (Rust CoreBPE) via Encoding.encode_ordinary_batch"
    except Exception:
        return None, None


def cpu_reference_run(pat, ranks, special, text, off, target_s, cores):
    """Time the reference CPU path on a bounded prefix of the workload (about target_s seconds).
    Returns (GB/s, Mtok/s, description dict)."""
    ref, how = load_reference_engine(pat, ranks, special)
    n_docs = len(off) - 1

    def docs_upto(nbytes):
        k = int(np.searchsorted(off, nbytes, side="right")) - 1
        k = max(1, min(k, n_docs))
        return k, int(off[k])

    if ref is not None:
        kind = "reference"

        def run(k):
            docs = [text[int(off[i]):int(off[i + 1])].tobytes().decode("utf-8") for i in range(k)]
            ref.encode("warmup")
            t0 = time.perf_counter()
            out = ref.encode_ordinary_batch(docs, num_threads=cores)
            dt = time.perf_counter() - t0
            return dt, sum(len(x) for x in out)
    else:
        from oracle import Oracle
        orc = Oracle(ranks, special, pat)
        kind, how = "port", "oracle/bpe_oracle.c (C restatement), pthread batch driver"

        def run(k):
            t0 = time.perf_counter()
            toks, _ = orc.encode_ordinary_batch_np(text[:int(off[k])], off[:k + 1], cores)
            return time.perf_counter() - t0, len(toks)

    k0, b0 = docs_upto(8 << 20)
    dt0, _ = run(k0)                                          # probe to size the sample
    rate = b0 / max(dt0, 1e-6)
    k, b = docs_upto(int(min(len(text), max(b0, rate * target_s))))
    dt, ntok = run(k)
    return b / dt / 1e9, ntok / dt / 1e6, {"kind": kind, "cores": cores, "how": how, "seconds": dt,
                                           "sample": f"first {k} docs = {b} bytes of the workload, {dt:.1f} s"}


class Bench:
    """One workload on this rank: corpus, engine, device buffers, and the three measurements."""

    def __init__(self, workload, nbytes, rank, world, local_rank, seed_offset=0, text_off=None):
        import torch
        import tiktoken_b200
        self.torch = torch
        self.workload, self.rank, self.world = workload, rank, world
        enc_name, builder, self.desc = WORKLOADS[workload]
        self.enc_name = enc_name
        self.pat, self.ranks, self.special, self.vocab_src = vu.load_encoding(enc_name)
        self.enc = tiktoken_b200.Encoding(f"{enc_name}_bench_{workload}", pat_str=self.pat, mergeable_ranks=self.ranks,
                                          special_tokens=self.special, device=local_rank)
        self.core = self.enc._core_bpe
        if text_off is None:
            text_off = builder(nbytes, SEEDS[workload] + seed_offset)
        self.text, self.off = text_off
        self.n_docs, self.N = len(self.off) - 1, len(self.text)
        # pinned host copies (the e2e path copies FROM these every step)
        self.h_text = torch.empty(max(self.N, 1), dtype=torch.uint8, pin_memory=True)
        self.h_text.numpy()[:self.N] = self.text
        self.h_off = torch.empty(self.n_docs + 1, dtype=torch.int64, pin_memory=True)
        self.h_off.numpy()[:] = self.off.astype(np.int64)
        self.stream = torch.cuda.Stream()                                       # a real (non-default) stream handle
        with torch.cuda.stream(self.stream):
            self.d_text = self.h_text.cuda(non_blocking=True)
            self.d_off = self.h_off.cuda(non_blocking=True)
            self.d_tok = torch.empty(max(self.N, 1), dtype=torch.int32, device="cuda")
            self.d_toff = torch.empty(self.n_docs + 1, dtype=torch.int64, device="cuda")
        self.stream.synchronize()

    # ---- one device-resident step, enqueue only
    def enqueue(self, counts_ptr=0):
        self.core.encode_device_async(self.d_text.data_ptr(), self.N, self.d_off.data_ptr(), self.n_docs,
                                      self.d_tok.data_ptr(), self.d_toff.data_ptr(), counts_ptr, self.stream.cuda_stream)

    def step_sync(self):
        self.enqueue()
        return self.core.device_wait()

    def parity(self, cores, sample_bytes=48 << 20):
        """Bit-exact check of the device-resident result against the oracle on a sample of whole documents starting at
        a rank-dependent place; the full result is then the reference for the e2e comparison."""
        from oracle import Oracle
        n_tok = self.step_sync()
        orc = Oracle(self.ranks, self.special, self.pat)
        off = self.off
        if self.n_docs == 1 or self.N <= sample_bytes:
            lo, hi = 0, self.n_docs
            if self.n_docs == 1 and self.N > (8 << 20):
                # one huge document: the oracle is single-threaded on it -- check a prefix cut at a line end as its own
                # document on BOTH sides (exact for the prefix because the cut is made the document end for both)
                cut = int(np.flatnonzero(self.text[:8 << 20] == 0x0A)[-1]) + 1
                sub_off = np.asarray([0, cut], np.uint64)
                buf = self.enc.encode_ordinary_packed(self.text[:cut], sub_off)
                exp_t, exp_o = orc.encode_ordinary_batch_np(self.text[:cut], sub_off, 1)
                ok = np.array_equal(buf.tokens(), exp_t) and np.array_equal(buf.offsets(), exp_o)
                buf.close()
                return ok, n_tok
        else:
            start = (self.rank * 0x9E3779B1 + 12345) % max(1, self.N - sample_bytes)
            lo = int(np.searchsorted(off, start, side="left"))
            hi = int(np.searchsorted(off, int(off[lo]) + sample_bytes, side="right")) - 1
            hi = max(lo + 1, min(hi, self.n_docs))
        b0, b1 = int(off[lo]), int(off[hi])
        exp_t, exp_o = orc.encode_ordinary_batch_np(self.text[b0:b1], (off[lo:hi + 1] - off[lo]).astype(np.uint64), cores)
        got_o = self.d_toff[lo:hi + 1].cpu().numpy().astype(np.uint64)
        got_t = self.d_tok[int(got_o[0]):int(got_o[-1])].cpu().numpy().view(np.uint32)
        ok = np.array_equal(got_o - got_o[0], exp_o) and np.array_equal(got_t, exp_t)
        return ok, n_tok

    def e2e(self, steps, compare=True):
        """Host pinned -> host pinned through the public API; returns (seconds per step, tokens, identical to the
        device-resident result?)."""
        torch = self.torch
        h_text_np, h_off_np = self.h_text.numpy()[:self.N], self.h_off.numpy().view(np.uint64)
        for _ in range(2):
            self.enc.encode_ordinary_packed(h_text_np, h_off_np).close()
        torch.cuda.synchronize()
        ts, same, ntok = [], True, 0
        for i in range(steps):
            t0 = time.perf_counter()
            buf = self.enc.encode_ordinary_packed(h_text_np, h_off_np)      # H2D + kernels + D2H, synchronous
            ts.append(time.perf_counter() - t0)
            ntok = buf.n_tokens
            if compare and i == 0:
                dev_t = self.d_tok[:ntok].cpu().numpy().view(np.uint32)
                dev_o = self.d_toff.cpu().numpy().astype(np.uint64)
                same = bool(np.array_equal(buf.tokens(), dev_t) and np.array_equal(buf.offsets(), dev_o))
            buf.close()
        return float(np.mean(ts)), ntok, same, self.core.last_timings()

    def dump_outputs(self, out_dir, n_tok, counts):
        """Write what the last device-resident step returned -- the tokens, the per-document token offsets and the
        {n_tokens, n_docs} counts its last kernel wrote -- as out_dir/<name>.npy in float64 (exact for these integers).
        Tokens and offsets are a fixed, seeded sample of positions, stored as <name>_positions.npy: under 59 MB in all
        (the 1 GiB config2 corpus encodes to over 200 M tokens)."""
        torch = self.torch
        os.makedirs(out_dir, exist_ok=True)
        arrays = {"counts": np.asarray(counts, np.float64)}
        for name, dev, n, k in (("tokens", self.d_tok, n_tok, 3 << 20), ("token_offsets", self.d_toff, self.n_docs + 1, 1 << 19)):
            pos = sample_positions(n, k)
            arrays[name] = dev[torch.from_numpy(pos).to(dev.device)].cpu().numpy().astype(np.float64)
            arrays[name + "_positions"] = pos.astype(np.float64)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)

    def close(self):
        del self.d_text, self.d_off, self.d_tok, self.d_toff, self.h_text, self.h_off, self.core, self.enc
        self.torch.cuda.empty_cache()


def timed_device_loop(b: Bench, steps, world, xchg):
    """K steps enqueued back to back on b.stream, one NCCL count exchange per step enqueued behind each pipeline;
    CUDA events on that stream; returns ms for the K steps (this rank)."""
    torch = b.torch
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(b.stream):
        ev0.record(b.stream)
        for _ in range(steps):
            b.enqueue(xchg.send_ptr())
            xchg.post_device()             # all-gather of (tokens, docs) from the device buffer the pipeline just filled
            if len(xchg._pending) >= xchg.depth - 1:
                xchg.wait()
        placements = xchg.drain()          # every exchange completes inside the timed region
        ev1.record(b.stream)
    n_tok = b.core.device_wait()
    b.stream.synchronize()
    return ev0.elapsed_time(ev1), n_tok, placements


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--bytes", type=int, default=0, help="override the per-rank corpus size (development)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the block with the other BASELINE configs")
    ap.add_argument("--no-extras", action="store_true", help="skip api / strong-scaling / one-process multi-GPU lines")
    ap.add_argument("--decode", action="store_true", help="also time the device decode of the produced tokens (next row)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    enc_name, builder, wl_desc = WORKLOADS[args.workload]
    nbytes = args.bytes or DEFAULT_BYTES[args.workload]
    cores = os.cpu_count() or 1

    def config_of(workload, nb, parallelism=None):
        e, _, d = WORKLOADS[workload]
        return {"workload": f"{workload}: {d}", "bytes_per_gpu": nb, "encoding": e, "seed": SEEDS[workload],
                "l2": "inputs (>= 64 MiB text per step, streamed once) exceed or equal the 126 MB L2; no reuse between steps",
                "parallelism": parallelism or f"doc-sharded x{world}"}

    # ---------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        pat, ranks, special, vocab_src = vu.load_encoding(enc_name)
        sample_cap = min(nbytes, 256 << 20)
        text, off = builder(sample_cap, SEEDS[args.workload])
        vals, toks, secs = [], [], []
        desc = None
        for i in range(args.warmup + args.steps):
            gbs, mts, desc = cpu_reference_run(pat, ranks, special, text, off, args.cpu_seconds, cores)
            if i >= args.warmup:
                vals.append(gbs); toks.append(mts); secs.append(desc["seconds"])
        v = float(np.mean(vals))
        config = config_of(args.workload, nbytes)
        config["vocab"] = f"{vocab_src} ({len(ranks)} mergeable ranks)"
        config["timed_sample"] = f"each step times a bounded prefix of the first {sample_cap} bytes of the workload (see cpu_baseline.sample); a rate"
        line = {"impl": "reference", "metric": "input_GB_per_s", "value": v, "unit": "GB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "mtokens_per_s": float(np.mean(toks)), "config": config,
                "cpu_baseline": {"value": v, "unit": "GB/s", **desc},
                "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- B200 arm
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: tiktoken_b200 has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local_rank)
    from tiktoken_b200.sharding import CountExchange, bind_to_gpu_numa
    numa = bind_to_gpu_numa(local_rank)          # before any pinned allocation: first touch on the GPU's node
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank0_section(tag, fn):
        """Run fn on rank 0 while the other ranks wait on the HOST (c10d store), not in an NCCL barrier: their GPUs stay
        idle, which matters when rank 0 drives all of them through the one-process engine."""
        barrier()
        if world == 1:
            fn()
            return
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                fn()
            finally:
                store.set(f"b200bench_{tag}", "done")
        else:
            store.wait([f"b200bench_{tag}"])
        barrier()

    def allmax(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(*xs):
        t = torch.tensor([int(x) for x in xs], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(v) for v in t.tolist()]

    def allok(flag):
        t = torch.tensor([0 if flag else 1], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item()) == 0

    def measure(b: Bench, steps, warmup, sample_clocks=False, dump_dir=None):
        """parity gate (every rank) -> value -> e2e (compared with the device result); returns a dict."""
        ok, n_tok = b.parity(cores)
        if not allok(ok):
            return {"parity": False, "error": "PARITY FAILURE against the oracle"}
        xchg = CountExchange(rank, world, device="cuda")
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()                                     # nvidia-smi needs a moment to come up: start it before the warm-up
        timed_device_loop(b, 1, world, xchg)                    # also warms the NCCL communicator and settles work-space sizes
        if sampler:
            for _ in range(100):                                # ... and wait (bounded) until it delivers
                if sampler.rows:
                    break
                time.sleep(0.02)
        t_warm = time.perf_counter()
        for _ in range(max(warmup - 1, 2)):
            timed_device_loop(b, 1, world, xchg)
        barrier()
        t0 = time.perf_counter()
        ms_total, n_tok, placements = timed_device_loop(b, steps, world, xchg)
        t1 = time.perf_counter()
        barrier()
        clocks = sampler.stop(t0, t1, t_warm) if sampler else None
        if dump_dir and rank == 0:                              # before anything else overwrites the step's outputs
            b.dump_outputs(dump_dir, n_tok, placements[-1][0])
        per_rank = [ms_total / steps]
        if world > 1:                                           # which rank set the pace (the MAX is what counts)
            t = torch.tensor([ms_total / steps], dtype=torch.float64, device="cuda")
            g = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(g, t)
            per_rank = [float(x.item()) for x in g]
        ms_step = allmax(ms_total) / steps
        tot_bytes, tot_tokens = allsum(b.N, n_tok)
        b.step_sync()                                           # one instrumented step for the per-stage events
        tm = b.core.last_timings()
        e2e_s, e2e_tokens, same, e2e_tm = b.e2e(steps)
        barrier()
        e2e_s = allmax(e2e_s)
        same = allok(same and e2e_tokens == n_tok)
        return {"parity": bool(same), "value": tot_bytes / (ms_step * 1e-3) / 1e9, "ms_per_step": ms_step,
                "mtokens_per_s": tot_tokens / (ms_step * 1e-3) / 1e6, "bytes": tot_bytes, "tokens": tot_tokens,
                "n_tok_rank": n_tok, "per_rank_ms_per_step": per_rank, "stage_ms": {k: v for k, v in tm.items() if k.endswith("_ms")}, "launches": tm["launches"],
                "e2e": {"value": tot_bytes / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(b.N + 8 * (b.n_docs + 1)),
                        "d2h_bytes_per_step": int(4 * e2e_tokens + 8 * (b.n_docs + 1)), "ms_per_step": e2e_s * 1e3,
                        "mtokens_per_s": tot_tokens / e2e_s / 1e6, "identical_to_device_result": bool(same),
                        "h2d_ms": e2e_tm["h2d_ms"], "d2h_ms": e2e_tm["d2h_ms"], "device_ms": e2e_tm["device_total_ms"]},
                "clocks": clocks, "counts_exchanged": [int(x) for x in placements[-1][0][:, 0]] if placements else None}

    b = Bench(args.workload, nbytes, rank, world, local_rank, seed_offset=7919 * rank)   # weak scaling: own corpus per rank
    m = measure(b, args.steps, args.warmup, sample_clocks=True, dump_dir=args.dump_outputs)
    if not m.get("parity"):
        if rank == 0:
            print(json.dumps({"error": m.get("error", "e2e result differs from the device-resident result"), "detail": m}))
        return 3
    N, n_tok, n_docs = b.N, m["n_tok_rank"], b.n_docs
    stage = m["stage_ms"]
    config = config_of(args.workload, nbytes)
    config["vocab"] = f"{b.vocab_src} ({len(b.ranks)} mergeable ranks)"
    config["numa"] = numa

    # ---- roofline of the dominant kernel, algorithmic bytes per launch (DESIGN.md 3)
    peak, peak_src = measured_peak()
    kern_ms = {"pretok_kernel": stage["pretok_ms"], "probe_kernel": stage["probe_ms"],
               "miss_sort+miss_kernel": stage["encode_ms"] - stage["probe_ms"], "scan+gather_kernel": stage["gather_ms"],
               "long-piece kernels": stage["long_ms"]}
    alg = {"pretok_kernel": N + N // 8 + N // 8,                      # text + doc mask read, piece mask written
           "probe_kernel": N + N // 8 + 4 * n_tok,                    # text + piece mask read, one 4-byte slot per piece written
           "miss_sort+miss_kernel": None, "scan+gather_kernel": 8 * n_tok + 8 * (n_docs + 1),   # slots read, tokens + doc offsets written
           "long-piece kernels": None}
    dominant = max((k for k in kern_ms if alg[k]), key=lambda k: kern_ms[k])
    achieved = alg[dominant] / (kern_ms[dominant] * 1e-3) / 1e9
    traffic = None
    prof = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get(dominant.split("+")[-1], {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    pipeline_alg = N + 4 * n_tok + 16 * (n_docs + 1)                    # SURVEY 8(d): text + tokens + both offset arrays
    dev_ms = stage["device_total_ms"]
    line = {
        "metric": "input_GB_per_s", "value": m["value"], "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
        "mtokens_per_s": m["mtokens_per_s"], "bytes_per_token": m["bytes"] / max(1, m["tokens"]),
        "n_docs_per_gpu": n_docs, "gpu_launches": m["launches"] * args.steps,
        "timing": "K async steps on one CUDA stream, events on that stream, no host sync inside a step; max over ranks",
        "parity": {"oracle_sample_every_rank": True, "e2e_identical_to_device_result": True},
        "per_rank_ms_per_step": m["per_rank_ms_per_step"],
        "stage_ms": stage, "kernel_ms": kern_ms,
        "roofline": {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg[dominant], "kernel_ms": kern_ms[dominant],
                     "per_kernel": {k: {"ms": kern_ms[k], "algorithmic_bytes": alg[k],
                                        "frac": (alg[k] / (kern_ms[k] * 1e-3) / 1e9 / peak) if alg[k] and kern_ms[k] > 0 else None}
                                    for k in kern_ms},
                     "pipeline": {"algorithmic_bytes": pipeline_alg, "achieved": pipeline_alg / (dev_ms * 1e-3) / 1e9,
                                  "frac": pipeline_alg / (dev_ms * 1e-3) / 1e9 / peak,
                                  "hbm_read_only_frac": N / (dev_ms * 1e-3) / 1e9 / peak, "device_ms": dev_ms}},
        "e2e": m["e2e"], "clocks": m["clocks"],
    }

    # ---- the calls a tiktoken user makes (host marshalling inside the timed region), rank 0 only
    if not args.no_extras and args.workload == "config2":
        def api_section():
            try:
                api = {}
                k, nb = b.n_docs, N                                         # the whole workload, like `e2e`
                pageable = b.text if b.text.flags["C_CONTIGUOUS"] else np.ascontiguousarray(b.text)   # ordinary (pageable) numpy memory
                poff = b.off.astype(np.uint64)

                def timed(fn, reps=3):
                    fn().close(); fn().close()                              # warm: staging blocks, pinned result of this size
                    ts = []
                    for _ in range(reps):
                        t0 = time.perf_counter(); buf = fn(); ts.append(time.perf_counter() - t0); buf.close()
                    return float(np.mean(ts))
                dt = timed(lambda: b.enc.encode_ordinary_packed(pageable, poff))
                api["packed_pageable"] = {"value": nb / dt / 1e9, "unit": "GB/s", "bytes": nb,
                                          "what": "encode_ordinary_packed(numpy in pageable memory): helper threads stage it into pinned "
                                                  "blocks by quarters + upload stream + kernels + D2H"}
                h_np = b.h_text.numpy()[:nb]
                dt = timed(lambda: b.enc.encode_packed(h_np, poff, allowed_special={"<|endoftext|>"}))
                api["encode_batch_default_policy_pinned"] = {
                    "value": nb / dt / 1e9, "unit": "GB/s", "bytes": nb,
                    "what": "encode_batch semantics (allowed {<|endoftext|>}, every other special disallowed = default policy) "
                            "on packed pinned input: device multi-pattern scan + pipeline, zero-copy pinned result"}
                docs = [bytes(b.text[int(b.off[i]):int(b.off[i + 1])]).decode("utf-8") for i in range(min(k, 1024))]
                dbytes = sum(len(d.encode()) for d in docs)
                b.enc.encode_ordinary_batch(docs)
                t0 = time.perf_counter()
                out = b.enc.encode_ordinary_batch(docs); dt = time.perf_counter() - t0
                api["list_str_to_list_list_int"] = {"value": dbytes / dt / 1e9, "unit": "GB/s", "bytes": dbytes, "docs": len(docs),
                                                    "what": "encode_ordinary_batch(list[str]) -> list[list[int]]: C marshalling both ways + device"}
                t0 = time.perf_counter()
                toks, offs = b.enc.encode_ordinary_batch_to_numpy(docs); dt = time.perf_counter() - t0
                api["list_str_to_numpy"] = {"value": dbytes / dt / 1e9, "unit": "GB/s", "bytes": dbytes,
                                            "what": "encode_ordinary_batch_to_numpy(list[str]) -> (tokens, offsets) arrays"}
                # latency of ONE small call (the whole pipeline is ~30 launches + one synchronisation, whatever the size)
                lat = {}
                for nbytes_small in (1 << 10, 64 << 10):
                    cut = int(np.flatnonzero(b.text[:nbytes_small] == 0x20)[-1])      # end the document at a space, not inside a scalar
                    small = np.ascontiguousarray(b.text[:cut]); soff = np.asarray([0, len(small)], np.uint64)
                    for _ in range(20):
                        b.enc.encode_ordinary_packed(small, soff).close()
                    t0 = time.perf_counter()
                    for _ in range(200):
                        b.enc.encode_ordinary_packed(small, soff).close()
                    lat[f"{nbytes_small >> 10}KiB_us"] = (time.perf_counter() - t0) / 200 * 1e6
                api["small_call_latency"] = dict(lat, what="encode_ordinary_packed of ONE document, host in -> host out, mean of 200 calls")
                del out, toks, offs, docs, pageable
                line["api"] = api
            except Exception as e:                                   # noqa: BLE001
                line["api"] = {"error": repr(e)}
        rank0_section("api", api_section)

    if args.decode and world == 1:
        h_text_np, h_off_np = b.h_text.numpy()[:N], b.h_off.numpy().view(np.uint64)
        buf = b.enc.encode_ordinary_packed(h_text_np, h_off_np)
        dtoks, doffs = np.array(buf.tokens()), np.array(buf.offsets())
        buf.close()
        b.enc.decode_packed(dtoks, doffs)
        dt = []
        for _ in range(3):
            t0 = time.perf_counter()
            data, boff = b.enc.decode_packed(dtoks, doffs)
            dt.append(time.perf_counter() - t0)
        assert len(data) == N
        line["decode"] = {"value": N / float(np.mean(dt)) / 1e9, "unit": "GB/s of decoded bytes (host tokens -> host bytes)",
                          "device_ms": b.core.last_timings()["device_total_ms"], "ms_per_step": float(np.mean(dt)) * 1e3}
    if not args.no_cpu_baseline and world == 1:
        gbs, mts, desc = cpu_reference_run(b.pat, b.ranks, b.special, b.text, b.off, args.cpu_seconds, cores)
        line["cpu_baseline"] = {"value": gbs, "unit": "GB/s", "mtokens_per_s": mts, **desc}
    b.close()
    del b

    # ---- strong scaling: ONE 1 GiB corpus (the same bytes whatever N), each rank a contiguous 1/N of it
    if not args.no_extras and args.workload == "config2" and not args.bytes:
        try:
            per = ((nbytes // world) // corpus.CHUNK) * corpus.CHUNK
            lo, hi = rank * per, (nbytes if rank == world - 1 else (rank + 1) * per)
            part = corpus.generate_range(corpus.ENGLISH, SEEDS["config2"], nbytes, lo, hi)
            bs = Bench("config2", hi - lo, rank, world, local_rank, text_off=corpus.docs_fixed(part, 65536, at_space=True))
            ms = measure(bs, args.steps, 2)
            line["strong"] = {"scaling": "strong", "total_bytes": ms.get("bytes"), "value": ms.get("value"), "unit": "GB/s",
                              "ms_per_step": ms.get("ms_per_step"), "parity": ms.get("parity"),
                              "e2e": {k: ms["e2e"][k] for k in ("value", "unit", "ms_per_step")} if ms.get("parity") else None,
                              "what": f"one {nbytes}-byte corpus (seed {SEEDS['config2']}) split into {world} contiguous shards"}
            bs.close()
            del bs
        except Exception as e:                                       # noqa: BLE001
            line["strong"] = {"error": repr(e)}

    # ---- the other BASELINE.json configs at their stated sizes (same method: parity gate, value, e2e)
    if not args.no_configs and args.workload == "config2" and not args.bytes:
        cfgs = {}
        for w in ("config3", "config4", "config5", "config1"):
            try:
                nb = DEFAULT_BYTES[w]
                single = w in ("config5", "config1")                 # one document: does not shard -> replicas (DESIGN 5)
                bw = Bench(w, nb, rank, world, local_rank, seed_offset=0 if single else 7919 * rank)
                mw = measure(bw, 3, 2)
                entry = {"config": config_of(w, nb, "replicas (one document cannot shard)" if single else None)}
                entry["config"]["vocab"] = f"{bw.vocab_src} ({len(bw.ranks)} mergeable ranks)"
                entry.update({k: mw.get(k) for k in ("parity", "value", "ms_per_step", "mtokens_per_s", "stage_ms", "error")})
                entry["unit"] = "GB/s"
                if mw.get("parity"):
                    entry["e2e"] = {k: mw["e2e"][k] for k in ("value", "unit", "ms_per_step", "identical_to_device_result")}
                    entry["n_docs_per_gpu"] = bw.n_docs
                if w == "config1" and rank == 0 and mw.get("parity"):
                    # plumbing line of BASELINE config 1: token count + sha256 of the uint32 array, GPU vs the reference on CPU
                    buf = bw.enc.encode_ordinary_packed(bw.text, bw.off)
                    got = np.array(buf.tokens()); buf.close()
                    ref, how = load_reference_engine(bw.pat, bw.ranks, bw.special)
                    t0 = time.perf_counter()
                    exp = np.asarray(ref.encode_ordinary(bw.text.tobytes().decode()), np.uint32) if ref is not None else None
                    dt = time.perf_counter() - t0
                    entry["plumbing"] = {"n_tokens": int(len(got)), "sha256_u32": hashlib.sha256(got.tobytes()).hexdigest(),
                                         "reference_cpu": how, "reference_sha256_u32": hashlib.sha256(exp.tobytes()).hexdigest() if exp is not None else None,
                                         "reference_cpu_seconds_1_thread": dt if exp is not None else None,
                                         "identical": bool(exp is not None and np.array_equal(got, exp))}
                cfgs[w] = entry
                bw.close()
                del bw
            except Exception as e:                                   # noqa: BLE001
                cfgs[w] = {"error": repr(e)}
        line["configs"] = cfgs

    # ---- ONE process driving every GPU of the job through the same C ABI (b200bpe_create_multi): rank 0, the others idle
    if not args.no_extras and args.workload == "config2" and world > 1 and not args.bytes:
        def multi_section():
            try:
                import tiktoken_b200
                pat, ranks, special, _ = vu.load_encoding("cl100k_base")
                encm = tiktoken_b200.Encoding("cl100k_multi", pat_str=pat, mergeable_ranks=ranks, special_tokens=special,
                                              devices=list(range(world)))
                text, off = corpus.config2(nbytes, SEEDS["config2"])
                h_text = torch.empty(len(text), dtype=torch.uint8, pin_memory=True); h_text.numpy()[:] = text
                off64 = off.astype(np.uint64)
                single = tiktoken_b200.Encoding("cl100k_single", pat_str=pat, mergeable_ranks=ranks, special_tokens=special, device=0)
                ref_buf = single.encode_ordinary_packed(h_text.numpy(), off64)
                encm.encode_ordinary_packed(h_text.numpy(), off64).close()
                ts = []
                for i in range(3):
                    t0 = time.perf_counter()
                    buf = encm.encode_ordinary_packed(h_text.numpy(), off64); ts.append(time.perf_counter() - t0)
                    if i == 0:
                        same = bool(np.array_equal(buf.tokens(), ref_buf.tokens()) and np.array_equal(buf.offsets(), ref_buf.offsets()))
                    buf.close()
                ref_buf.close()
                line["one_process_multi_gpu"] = {"devices": world, "value": len(text) / float(np.mean(ts)) / 1e9, "unit": "GB/s",
                                                 "ms_per_step": float(np.mean(ts)) * 1e3, "identical_to_single_gpu_result": same,
                                                 "what": "Encoding(devices=[0..N-1]).encode_ordinary_packed on ONE 1 GiB pinned corpus, one process"}
                del encm, single
            except Exception as e:                                   # noqa: BLE001
                line["one_process_multi_gpu"] = {"error": repr(e)}
        rank0_section("multi", multi_section)

    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
