#!/usr/bin/env python3
"""bench.py -- the openclaw-governance hot path on B200: messages scanned / s.

One *step* = one pass of the scan hot path (gram filter + exact factors, resolve, exact verification, result words)
over one batch of synthetic messages.  Workload at N=1: BASELINE.json configs[1] -- 1 M synthetic 256-byte messages x
500-rule firewall scan; for N>1 every rank scans its own 1 M-message shard (weak scaling; no data-path collective for
the scan).  The traffic is drawn from a 64 K-word vocabulary in which 2 % of the words are prefixes / suffixes of the
rule set's own literals; nothing in the library is tuned on data (the filter is compiled from the rules alone), and the
line carries the other vocabularies / hit rates / rule counts as extra.variants.  The JSON line also carries
  roofline     : achieved algorithmic HBM GB/s of the scan kernel (n*(L+12) bytes per launch,
                 SURVEY 8(d)) against MEASURED_PEAKS.json, measured live with CUDA events
  cpu_baseline : the CPU oracle port (oracle/, kind "port") on the box's host cores, a strided sample of the SAME batch
                 (also the parity check of the timed batch: result words equal)
  e2e          : the same metric through the C ABI with HOST (pinned) buffers, copies inside
  extra.merkle : Proof-of-Guardrails Merkle leaves/s (C3: 16 Mi x 256 B leaves per rank), block roots
                 all-gathered over NCCL and folded (the one collective on this path); root checked against the oracle
  extra.c4     : BASELINE configs[3]: 10 M messages split over the ranks (strong scaling) + the Merkle tree over the
                 event log of that very scan (one 32-byte record per message), one all-gather of shard roots
`--impl reference` times the reference path's CPU restatement (Node.js is not in this image or on
the GPU box, and the reference has no native sources to compile, so oracle/ is the only runnable
form of it) on all host threads.
`--dump-outputs DIR` writes the result words of the last timed step (rank 0) to DIR/scan_words.npy: the inputs are seeded,
so two builds of the project run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_MSGS = 1 << 20
MSG_LEN = 256
N_RULES = 500
P_HIT = 0.01
VOCAB_WORDS = 1 << 16      # headline traffic: 64 K-word vocabulary,
FRAG_FRAC = 0.02           # 2 % of its words are prefixes / suffixes of rule literals
C4_MSGS = 10_000_000
MERKLE_LEAVES = 1 << 24
MERKLE_LEAF = 256
MERKLE_BLOCK_LOG2 = 16
DUMP_MAX_BYTES = 64_000_000


def dump_scan_words(out_dir, words):
    """--dump-outputs: the result words a caller of the timed path receives (uint64 per message: hit << 63 |
    #rules hit << 32 | lowest hit rule) as DIR/scan_words.npy, float64 [k, 3] = (message index, high 32 bits, low 32
    bits), exact in float64.  Batches whose rows exceed DUMP_MAX_BYTES are sampled at fixed, seeded message indices."""
    words = np.ascontiguousarray(words).view(np.uint64)
    n = len(words)
    cap = (DUMP_MAX_BYTES - 4096) // (3 * 8)
    idx = np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
    w = words[idx]
    table = np.stack([idx.astype(np.float64), (w >> np.uint64(32)).astype(np.float64), (w & np.uint64(0xFFFFFFFF)).astype(np.float64)], axis=1)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scan_words.npy"), table)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: an in-process NVML poll every ~0.5 ms between
    start (construction) and stop() -- the region is only a few milliseconds long, an `nvidia-smi -lms` child would
    mostly report the idle GPU after it.  Falls back to one nvidia-smi query if NVML is unavailable."""

    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("hw_power_brake", 0x80))

    def __init__(self, index: int):
        import threading
        self.samples, self.reasons, self.max_mhz, self._stop, self.t = [], set(), None, False, None
        self.index = index
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            h = None
            try:
                pr = torch.cuda.get_device_properties(index)
                bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
                h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM); pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)   # first calls are slow: not inside the region

            def loop():
                k = 0
                while not self._stop:
                    try:
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        if k % 3 == 0:
                            r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                            for name, bit in self.REASONS:
                                if r & bit:
                                    self.reasons.add(name)
                    except Exception:
                        pass
                    k += 1
                    time.sleep(0.0003)
            self.t = threading.Thread(target=loop, daemon=True)
            self.t.start()
        except Exception:
            self.t = None

    def stop(self):
        if self.t is None:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip().split(",")
                return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [], "samples": 1, "source": "nvidia-smi after the region (NVML unavailable)"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"], "samples": 0}
        self._stop = True
        self.t.join(timeout=2)
        sm = self.samples
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(sm),
                "source": "NVML polled inside the timed region"}


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def find_node():
    """Is there a Node.js on this box?  (the reference's own runtime; BASELINE.md section 3)"""
    import glob
    import shutil
    for c in ("node", "nodejs"):
        pth = shutil.which(c)
        if pth:
            return pth
    for pat in ("~/.nvm/versions/node/*/bin/node", "/usr/local/bin/node", "/usr/lib/node_modules/../../bin/node", os.path.join(ROOT, "baseline", "_ref", "bin", "node")):
        for pth in glob.glob(os.path.expanduser(pat)):
            if os.access(pth, os.X_OK):
                return pth
    return None


def reference_arm(args, rank, world, emit=None):
    """The reference's own CPU implementation of the path, restated (oracle/): policy-semantics scan
    (matchesAny: RegExp.test per rule, gov/src/conditions/context.ts:9-25) on every CPU this process may use, threads
    pinned.  Every step scans the same fixed-size strided sample of the headline batch."""
    if rank != 0:
        return
    from oracle import oracle as O
    from vainplex_openclaw_b200 import workload as W
    rl = W.make_rules(N_RULES)
    regs = [O.Regex(r["source"], "i" if r["flags"] else "") for r in rl]
    threads = host_threads()
    sample = int(os.environ.get("CG_REF_SAMPLE", 16384))          # the same sample on every box, whatever its speed
    data_t, off_t, _ = W.make_messages(sample, MSG_LEN, rl, p_hit=P_HIT, seed=W.SEED_MSG, vocab_seed=W.SEED_MSG, vocab_words=VOCAB_WORDS, frag_frac=FRAG_FRAC)
    data, off = data_t.numpy(), off_t.numpy().astype(np.uint64)
    O.scan_policy(regs, data[: 1024 * MSG_LEN + 64], off[:1025], threads=threads, want_bits=False)       # untimed: page in, spawn threads
    for _ in range(min(args.warmup, 2)):
        O.scan_policy(regs, data, off, threads=threads, want_bits=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, words = O.scan_policy(regs, data, off, threads=threads, want_bits=False)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_scan_words(args.dump_outputs, words)
    v = sample * args.steps / dt
    node = find_node()
    line = {"metric": "messages_scanned_per_s", "value": v, "unit": "msgs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": "1M x 256B msgs x 500 rules (C2), policy semantics; fixed sample of %d msgs per step" % sample,
                       "rules": N_RULES, "msg_len": MSG_LEN},
            "cpu_baseline": {"value": v, "unit": "msgs/s", "cores": threads, "per_core": v / threads, "kind": "port",
                             "sample": "%d messages x %d rules per step, oracle/jsre.c backtracking matcher (-O3), %d pinned threads = the process's CPU affinity (os.cpu_count() = %s); "
                                       "Node.js on this box: %s -- restated oracle, not Node" % (sample, N_RULES, threads, os.cpu_count(), node or "not found")},
            "e2e": {"value": v, "unit": "msgs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    (emit or (lambda o: print(json.dumps(o))))(line)


def main():
    # stdout carries exactly ONE JSON line: anything a library prints on fd 1 meanwhile (NCCL's version banner, ...)
    # goes to stderr instead; the real stdout is restored for the final print
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--msgs", type=int, default=N_MSGS)
    ap.add_argument("--len", type=int, default=MSG_LEN, dest="msg_len")
    ap.add_argument("--rules", type=int, default=N_RULES)
    ap.add_argument("--stride", type=int, default=0, help="gram filter stride: 0 = the compiler's choice, 2 or 4")
    ap.add_argument("--p-hit", type=float, default=None, help="fraction of messages with an injected rule-matching token (default 0.01; SURVEY 8d also names 0 and 0.10)")
    ap.add_argument("--seed-offset", type=int, default=0, help="shift the synthetic data seed and vocabulary")
    ap.add_argument("--vocab", type=int, default=VOCAB_WORDS, help="words in the traffic's vocabulary")
    ap.add_argument("--frag-frac", type=float, default=FRAG_FRAC, help="fraction of vocabulary words that are prefixes / suffixes of rule literals")
    ap.add_argument("--no-merkle", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--merkle-leaves", type=int, default=MERKLE_LEAVES)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result words of the last one to DIR/scan_words.npy (see dump_scan_words)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global P_HIT
    if args.p_hit is not None:
        P_HIT = args.p_hit
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return reference_arm(args, rank, world, emit)

    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
    import torch
    import torch.distributed as dist
    from vainplex_openclaw_b200 import _native as N, sharding, workload as W
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N.init(local)
    n, L, R = args.msgs, args.msg_len, args.rules
    rl = W.make_rules(R)
    rules = W.rules_as_tuples(rl)
    t0 = time.perf_counter()
    rs = N.Ruleset(rules, options=args.stride, strict=True)
    compile_s = time.perf_counter() - t0
    info = rs.info()
    stream = torch.cuda.Stream(device=dev)          # a real (non-default) stream: handle 0 would mean "library stream" to the C ABI
    peak, peak_src = measured_peaks()

    def gen(nmsgs, ruleset_rl, p_hit, seed_off, vocab, frag):
        # ranks of one run share the vocabulary (the "language" of the traffic) and draw different messages
        d, o64, injected = W.make_messages(nmsgs, L, ruleset_rl, p_hit=p_hit, seed=W.SEED_MSG + rank + seed_off, device=dev,
                                            vocab_seed=W.SEED_MSG + seed_off, vocab_words=vocab, frag_frac=frag)
        return d, o64.to(torch.int32), injected        # uint32 offsets (bit pattern) as the C ABI expects; n*L < 2^31 here

    def measure(ruleset, d, o, nmsgs, steps, warmup, profile_steps):
        """-> (ms_per_step over `steps` graph-replayed steps, per-kernel ms medians, counters, result words of the last timed step,
        whether every timed step's words equal the profiled step's)"""
        outs = [torch.zeros(nmsgs, dtype=torch.int64, device=dev) for _ in range(2)]
        k = [0]

        def step():
            ruleset.scan_batch_device(d.data_ptr(), o.data_ptr(), nmsgs, outs[k[0] & 1].data_ptr(), stream.cuda_stream)
            k[0] += 1
        with torch.cuda.stream(stream):
            for attempt in range(8):                # warm-up; a queue that overflows is reported once by scan_join, the library
                for _ in range(warmup):             # has grown the scratch by then: scan again (the device-path contract, openclaw_gov.h)
                    step()
                try:
                    ruleset.scan_join(stream.cuda_stream)
                    break
                except N.GovError as e:
                    if e.code != N.CG_ERR_CAPACITY or attempt == 7:
                        raise
            N.set_profiling(True)                   # kernel breakdown: events inside the library, one sync per step (not the headline timing)
            kms = []
            for _ in range(profile_steps):
                step(); torch.cuda.synchronize(); kms.append(N.last_kernel_ms() + N.last_tail_ms())
            N.set_profiling(False)
            ruleset.scan_join(stream.cuda_stream)
            counters = ruleset.work_counters()
            ref_words = outs[(k[0] - 1) & 1].clone()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                step()
            e1.record(stream)
            ruleset.scan_join(stream.cuda_stream)        # waits for the stream; raises if a batch overflowed a queue
            torch.cuda.synchronize()
        same = bool(torch.equal(outs[0], ref_words) and torch.equal(outs[1], ref_words))
        return e0.elapsed_time(e1) / steps, np.median(np.array(kms), axis=0), counters, outs[(k[0] - 1) & 1], same

    # ---- headline: K steps, device-resident inputs (256 MiB per step > 126 MB L2), barrier + sync both sides
    data, off, inj = gen(n, rl, P_HIT, args.seed_offset, args.vocab, args.frag_frac)
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = N.launch_count()
    ms_local, kms, counters, words, steps_equal = measure(rs, data, off, n, args.steps, args.warmup, min(args.steps, 10))
    launches_total = N.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    launches = int(round(launches_total * args.steps / float(args.steps + args.warmup + min(args.steps, 10))))     # kernels of the timed steps only
    per_rank_ms = [ms_local]
    ms_per_step = ms_local
    if world > 1:
        t = torch.tensor([ms_local], device=dev, dtype=torch.float64)
        allt = torch.zeros(world, device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(allt, t)
        per_rank_ms = [float(x) for x in allt.tolist()]
        ms_per_step = float(allt.max().item())
        dist.barrier()
    value = world * n / (ms_per_step * 1e-3)
    scan_ms = float(kms[0])
    alg_bytes = n * (L + 12)

    # ---- e2e through the host-buffer C ABI call: pinned host input -> H2D -> kernels -> D2H words
    h_data = torch.empty(data.numel(), dtype=torch.uint8, pin_memory=True); h_data.copy_(data)
    h_off = torch.empty(n + 1, dtype=torch.int32, pin_memory=True); h_off.copy_(off)
    h_words = torch.empty(n, dtype=torch.int64, pin_memory=True)
    import ctypes as C
    lib = N.load()
    nh = C.c_uint32(0)

    def e2e_step():
        N.check(lib.cg_scan_batch(rs.handle, h_data.data_ptr(), h_off.data_ptr(), n, h_words.data_ptr(), None, 0, C.byref(nh)))

    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        e2e_step()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * n * e2e_steps / e2e_s
    same = bool(torch.equal(h_words.to(dev), words))

    # ---- the other workloads of SURVEY 8(d), each a short device-resident run of its own (N = 1 only; rank 0 of a multi-GPU
    # run skips them: they say nothing about scaling)
    variants = None
    if world == 1 and not args.no_variants:
        variants = {}

        def variant(name, nrules=R, p_hit=P_HIT, seed_off=args.seed_offset, vocab=args.vocab, frag=args.frag_frac, nmsgs=n):
            vrl = rl if nrules == R else W.make_rules(nrules)
            vrs = rs if nrules == R else N.Ruleset(W.rules_as_tuples(vrl), options=args.stride, strict=True)
            d, o, _ = gen(nmsgs, vrl, p_hit, seed_off, vocab, frag)
            ms, vk, vc, _, _ = measure(vrs, d, o, nmsgs, 6, 3, 3)
            variants[name] = {"rules": nrules, "p_hit": p_hit, "vocab_words": vocab, "frag_frac": frag, "ms_per_step": ms, "msgs_per_s": nmsgs / (ms * 1e-3),
                              "scan_ms": float(vk[0]), "tail_ms": {"confirm_kernel": float(vk[4]), "resolve_kernel": float(vk[5]), "verify": float(vk[2]), "finalize": float(vk[3])}, "scan_roofline_frac": nmsgs * (L + 12) / (float(vk[0]) * 1e-3) / 1e9 / peak,
                              "flagged_grams": vc[6], "confirmed_factor_occurrences": vc[4], "vm_pairs": vc[1], "stride": int(vrs.info().stride)}
            if vrs is not rs:
                vrs.close()
            del d, o
        variant("p_hit_0", p_hit=0.0)
        variant("p_hit_10pct", p_hit=0.10)
        variant("other_vocabulary", seed_off=args.seed_offset + 1)
        variant("random_4k_vocabulary_no_fragments", vocab=4096, frag=0.0)
        variant("fragments_10pct", frag=0.10)
        variant("rules_5000", nrules=5000)
        variant("rules_17_builtins", nrules=17)

    # C1: one message through the blocking single-message entry point (the synchronous hooks' path), 17 built-in rules
    one = None
    if world == 1:
        rs17 = N.Ruleset(W.rules_as_tuples(W.make_rules(17)), strict=True)
        m1 = bytes(h_data.numpy()[:L])
        tok = b"please use key sk-" + b"a" * 24 + b" for bob@example.com"
        for _ in range(20):
            rs17.scan_one(m1)
        t0 = time.perf_counter()
        for _ in range(200):
            rs17.scan_one(m1)
        lat = (time.perf_counter() - t0) / 200
        w1, r1 = rs17.scan_one(tok)
        one = {"latency_us": lat * 1e6, "rules": 17, "msg_bytes": L, "hit_rules_of_probe": r1}
        rs17.close()
    # (f1) redacted output through cg_redact_batch (findMatches semantics + digests + splice on the device), host buffers
    redact = None
    if world == 1:
        nr = min(n, 1 << 18)
        hd, ho = h_data.numpy()[: nr * L + 64], h_off.numpy()[: nr + 1].view(np.uint32)
        rs.redact_batch(hd, ho)
        t0 = time.perf_counter()
        r_out, r_off, r_spans, r_dig = rs.redact_batch(hd, ho)
        dt = time.perf_counter() - t0
        redact = {"msgs": nr, "msgs_per_s_from_host": nr / dt, "spans": int(len(r_spans)), "out_bytes": int(len(r_out)), "in_bytes": int(nr * L)}

    def merkle_of(leaves, leaf_len, nl, steps):
        """block roots of this rank's leaves -> all-gather (the one collective on this path) -> fold on every rank.
        -> (ms per tree (max over ranks), root bytes, this rank's block roots [nblk, 32] on the host)"""
        nblk = (nl + (1 << MERKLE_BLOCK_LOG2) - 1) >> MERKLE_BLOCK_LOG2
        # equal block counts per rank keep the all-gather rectangular; the fold skips nothing because blocks are aligned
        roots = torch.zeros(nblk * 32, dtype=torch.uint8, device=dev)
        allroots = torch.zeros(world * nblk * 32, dtype=torch.uint8, device=dev)
        root = torch.zeros(32, dtype=torch.uint8, device=dev)

        def merkle_step():
            N.check(lib.cg_merkle_block_roots_device(leaves.data_ptr(), leaf_len, nl, MERKLE_BLOCK_LOG2, roots.data_ptr(), stream.cuda_stream))
            if world > 1:
                dist.all_gather_into_tensor(allroots, roots)
            else:
                allroots.copy_(roots)
            N.check(lib.cg_merkle_fold_device(allroots.data_ptr(), world * nblk, root.data_ptr(), stream.cuda_stream))
        with torch.cuda.stream(stream):
            for _ in range(2):
                merkle_step()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            m0.record(stream)
            for _ in range(steps):
                merkle_step()
            m1.record(stream)
            torch.cuda.synchronize()
        mms = m0.elapsed_time(m1) / steps
        if world > 1:
            t = torch.tensor([mms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            mms = float(t.item())
        return mms, bytes(root.cpu().numpy()), roots.cpu().numpy().reshape(nblk, 32), allroots.cpu().numpy().reshape(world * nblk, 32)

    def oracle_block_roots_equal(h_leaves, leaf_len, nl, my_roots, all_roots, root):
        """this rank's block roots against the oracle over its own leaves (every rank checks its shard, threaded), and the
        fold of ALL gathered roots against the oracle's fold: together the N-rank root is oracle-checked"""
        from oracle import oracle as O
        from concurrent.futures import ThreadPoolExecutor
        B = 1 << MERKLE_BLOCK_LOG2
        nblk = my_roots.shape[0]
        th = max(1, host_threads() // max(1, world))

        def blk(b):
            cnt = min(B, nl - b * B)
            return O.merkle_root_fixed(h_leaves[b * B * leaf_len:], leaf_len, cnt) == my_roots[b].tobytes()
        with ThreadPoolExecutor(th) as ex:
            ok_blocks = all(ex.map(blk, range(nblk)))
        ok_fold = O.merkle_fold(all_roots) == root
        ok = bool(ok_blocks and ok_fold)
        if world > 1:
            t = torch.tensor([1 if ok else 0], device=dev, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok = bool(int(t.item()))
        return ok

    # ---- Merkle (C3): leaves/s; block roots all-gathered over NCCL, folded on every rank; root checked against the oracle
    merkle = None
    if not args.no_merkle:
        nl = args.merkle_leaves
        leaves = W.make_leaves(nl, MERKLE_LEAF, seed=W.SEED_LEAVES + rank, device=dev)
        mms, root, my_roots, all_roots = merkle_of(leaves, MERKLE_LEAF, nl, 5)
        t0 = time.perf_counter()
        h_leaves = leaves.cpu().numpy()
        root_ok = oracle_block_roots_equal(h_leaves, MERKLE_LEAF, nl, my_roots, all_roots, root)
        check_s = time.perf_counter() - t0
        nblk = my_roots.shape[0]
        # the same tree with the exchange INSIDE the library (cg_comm_init + cg_merkle_root_sharded_device: NCCL all-gather issued
        # by the C ABI, bound with dlopen); the id travels over the launcher's process group
        lib_coll = None
        try:
            if world > 1:
                ids = [N.comm_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(ids, src=0)
                N.comm_init(rank, world, ids[0])
            lroot = N.merkle_root_sharded_device(leaves.data_ptr(), MERKLE_LEAF, nl, world * nl, MERKLE_BLOCK_LOG2, stream.cuda_stream)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            tl = time.perf_counter()
            for _ in range(3):
                lroot = N.merkle_root_sharded_device(leaves.data_ptr(), MERKLE_LEAF, nl, world * nl, MERKLE_BLOCK_LOG2, stream.cuda_stream)
            lms = (time.perf_counter() - tl) / 3 * 1e3
            if world > 1:
                t = torch.tensor([lms], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); lms = float(t.item())
            lib_coll = {"ms_per_tree_host_clock": lms, "leaves_per_s": world * nl / (lms * 1e-3), "root_equals_the_other_path": lroot == root,
                        "collective": "ncclAllGather issued by libopenclaw_gov.so (cg_merkle_root_sharded_device)" if world > 1 else "none (1 rank)"}
        except Exception as e:       # noqa: BLE001 -- reported, the torch.distributed path above stays the headline
            lib_coll = {"error": str(e)[:200]}
        merkle = {"leaves_per_s": world * nl / (mms * 1e-3), "ms_per_tree": mms, "leaves_per_rank": nl, "leaf_bytes": MERKLE_LEAF,
                  "root_hex": root.hex(), "root_equals_oracle": root_ok,
                  "root_check": "every rank: its %d block roots == oracle over its own %d leaves; fold of all %d gathered roots == oracle fold (%.1f s on the host)" % (nblk, nl, world * nblk, check_s),
                  "collective": "all_gather of %d block roots/rank (NCCL)" % nblk if world > 1 else "none (1 rank)",
                  "library_collective": lib_coll,
                  "hbm_frac_of_measured": (nl * MERKLE_LEAF / (mms * 1e-3)) / (peak * 1e9),
                  "sha256_compressions_per_s": world * (nl * ((MERKLE_LEAF + 1 + 9 + 63) // 64) + 2 * (nl - 1)) / (mms * 1e-3)}
        # (f2) the append-only log fed from PINNED host memory (H2D inside the timed region), rank 0, N = 1 only:
        #      ragged leaves (JSONL-line-like lengths 64..320 B) in 16 appends; then the same bytes as one JSONL buffer
        #      split at '\n' on the device; consistency proof between the half-way tree and the final one
        if world == 1 and rank == 0:
            from oracle import oracle as O
            nlog = min(nl, 1 << 22)
            rngl = np.random.default_rng(4242)
            lens = rngl.integers(64, 321, nlog).astype(np.uint64)
            offs_all = np.zeros(nlog + 1, dtype=np.uint64); offs_all[1:] = np.cumsum(lens)
            total = int(offs_all[-1])
            src = leaves[:total + 64].clone()
            nlpos = torch.from_numpy((offs_all[1:] - 1).astype(np.int64)).to(src.device)
            src[nlpos] = 10                                    # every leaf ends in '\n' (and holds none elsewhere: make_leaves' alphabet)
            h_pin = torch.empty(total + 64, dtype=torch.uint8).pin_memory(); h_pin.copy_(src[:total + 64].cpu())
            o_pin = torch.empty(nlog + 1, dtype=torch.int64).pin_memory(); o_pin.copy_(torch.from_numpy(offs_all.astype(np.int64)))
            per = nlog // 16
            lg = N.MerkleLog(keep_leaf_digests=True)
            lg.append([b"warm-up"]); lg.close()
            lg = N.MerkleLog(keep_leaf_digests=True)
            lg.reserve(16 * per, total)                        # (the day's expected volume: no device reallocation inside the appends)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for c in range(16):
                # offsets are absolute into the one pinned buffer (the library copies bytes[offsets[0], offsets[m]))
                N.check(lib.cg_merkle_log_append(lg.handle, h_pin.data_ptr(), o_pin.data_ptr() + 8 * c * per, per))
                if c == 7:
                    half_root = lg.root()
            log_root = lg.root()
            dt = time.perf_counter() - t0
            t1 = time.perf_counter(); path = lg.proof(nlog // 3); proof_ms = (time.perf_counter() - t1) * 1e3
            t1 = time.perf_counter(); cons = lg.consistency(8 * per); cons_ms = (time.perf_counter() - t1) * 1e3
            h_np = h_pin.numpy()
            one_shot = N.merkle_root(h_np, offs_all[:16 * per + 1])
            leaf3 = bytes(h_np[int(offs_all[nlog // 3]):int(offs_all[nlog // 3 + 1])])
            # the same bytes as a day file: one buffer, split on the device (leaves = lines WITHOUT their '\n')
            lj = N.MerkleLog(keep_leaf_digests=False)
            t1 = time.perf_counter()
            kl = C.c_uint64(0)
            N.check(lib.cg_merkle_log_append_jsonl(lj.handle, h_pin.data_ptr(), int(offs_all[16 * per]), C.byref(kl)))
            jroot = lj.root(); dj = time.perf_counter() - t1
            sample = min(16 * per, 1 << 16)                    # oracle over a prefix (lines without '\n'), against the same prefix through the library
            so = np.zeros(sample + 1, dtype=np.uint64); so[1:] = np.cumsum(lens[:sample] - 1)
            sb = np.concatenate([h_np[int(offs_all[i]):int(offs_all[i + 1]) - 1] for i in range(sample)] + [np.zeros(64, dtype=np.uint8)])
            ls = N.MerkleLog(keep_leaf_digests=False); ls.append_jsonl(h_np[:int(offs_all[sample])]); sroot = ls.root(); ls.close()
            merkle["log"] = {"leaves": 16 * per, "appends": 16, "leaf_bytes": "ragged 64..320 (mean %.0f)" % float(lens.mean()), "host_memory": "pinned",
                             "leaves_per_s_from_host": 16 * per / dt, "GBps_from_host": int(offs_all[16 * per]) / dt / 1e9,
                             "root_equals_one_shot_tree": log_root == one_shot,
                             "proof_len": len(path), "proof_ms": proof_ms, "proof_verifies": N.merkle_verify_proof(leaf3, nlog // 3, 16 * per, path, log_root),
                             "consistency_len": len(cons), "consistency_ms": cons_ms,
                             "consistency_verifies": N.merkle_verify_consistency(8 * per, 16 * per, half_root, log_root, cons) and O.merkle_verify_consistency(8 * per, 16 * per, half_root, log_root, cons),
                             "jsonl": {"lines": int(kl.value), "bytes": int(offs_all[16 * per]), "lines_per_s_from_host": kl.value / dj,
                                       "prefix_root_equals_oracle": sroot == O.merkle_root(sb, so), "prefix_lines": sample}}
            lg.close(); lj.close()
            del src, h_pin, o_pin
        del leaves, h_leaves

    # ---- C4 (BASELINE configs[3]): 10 M messages split over the ranks + the Merkle tree over the event log of THAT scan
    # (one 32-byte record per message: global index, result word, first 16 message bytes), scan and tree on the same stream,
    # one all-gather of block roots.  Strong scaling: the total is fixed, value = 10 M / max-over-ranks time.
    c4 = None
    if not args.no_c4:
        lo, hi = sharding.shard_range(C4_MSGS, rank, world, align=1 << MERKLE_BLOCK_LOG2)
        nc = hi - lo
        nc_max = max(sharding.shard_range(C4_MSGS, r, world, align=1 << MERKLE_BLOCK_LOG2)[1] - sharding.shard_range(C4_MSGS, r, world, align=1 << MERKLE_BLOCK_LOG2)[0] for r in range(world))
        d4, o4, _ = gen(nc, rl, P_HIT, args.seed_offset + 7, args.vocab, args.frag_frac)
        w4 = torch.zeros(nc, dtype=torch.int64, device=dev)
        idx = torch.arange(lo, hi, dtype=torch.int64, device=dev)
        log = torch.zeros(nc_max * 32, dtype=torch.uint8, device=dev)          # (padded to the largest shard: equal block counts per rank)
        nblk4 = (nc_max + (1 << MERKLE_BLOCK_LOG2) - 1) >> MERKLE_BLOCK_LOG2
        roots4 = torch.zeros(nblk4 * 32, dtype=torch.uint8, device=dev)
        all4 = torch.zeros(world * nblk4 * 32, dtype=torch.uint8, device=dev)
        root4 = torch.zeros(32, dtype=torch.uint8, device=dev)
        nblk_mine = (nc + (1 << MERKLE_BLOCK_LOG2) - 1) >> MERKLE_BLOCK_LOG2
        msg_head = d4[: nc * L].view(nc, L)[:, :16]

        def c4_step():
            rs.scan_batch_device(d4.data_ptr(), o4.data_ptr(), nc, w4.data_ptr(), stream.cuda_stream)
            rec = log[: nc * 32].view(nc, 32)
            rec[:, 0:8] = idx.view(torch.uint8).view(nc, 8)
            rec[:, 8:16] = w4.view(torch.uint8).view(nc, 8)
            rec[:, 16:32] = msg_head
            roots4.zero_()
            N.check(lib.cg_merkle_block_roots_device(log.data_ptr(), 32, nc, MERKLE_BLOCK_LOG2, roots4.data_ptr(), stream.cuda_stream))
            if world > 1:
                dist.all_gather_into_tensor(all4, roots4)
            else:
                all4.copy_(roots4)
        with torch.cuda.stream(stream):
            for attempt in range(8):                # (warm-up; see measure(): an overflowing queue is reported once, then the scratch has grown)
                for _ in range(3):
                    c4_step()
                try:
                    rs.scan_join(stream.cuda_stream)
                    break
                except N.GovError as e:
                    if e.code != N.CG_ERR_CAPACITY or attempt == 7:
                        raise
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c4_steps = 5
            e0.record(stream)
            for _ in range(c4_steps):
                c4_step()
            e1.record(stream)
            rs.scan_join(stream.cuda_stream)
            torch.cuda.synchronize()
        c4_ms = e0.elapsed_time(e1) / c4_steps
        if world > 1:
            t = torch.tensor([c4_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            c4_ms = float(t.item())
        # the global root: the ranks' real block roots in shard order (shards are block-aligned, only the last one is ragged)
        counts = [((sharding.shard_range(C4_MSGS, r, world, align=1 << MERKLE_BLOCK_LOG2)[1] - sharding.shard_range(C4_MSGS, r, world, align=1 << MERKLE_BLOCK_LOG2)[0]) + (1 << MERKLE_BLOCK_LOG2) - 1) >> MERKLE_BLOCK_LOG2 for r in range(world)]
        allh = all4.cpu().numpy().reshape(world, nblk4, 32)
        real = np.concatenate([allh[r, :counts[r]] for r in range(world)], axis=0)
        real_d = torch.from_numpy(real.reshape(-1).copy()).to(dev)
        N.check(lib.cg_merkle_fold_device(real_d.data_ptr(), real.shape[0], root4.data_ptr(), stream.cuda_stream))
        torch.cuda.synchronize()
        from oracle import oracle as O
        h_log = log[: nc * 32].cpu().numpy()
        mine = allh[rank, :nblk_mine]
        ok4 = all(O.merkle_root_fixed(h_log[b * (1 << MERKLE_BLOCK_LOG2) * 32:], 32, min(1 << MERKLE_BLOCK_LOG2, nc - b * (1 << MERKLE_BLOCK_LOG2))) == mine[b].tobytes() for b in range(nblk_mine))
        ok4 = ok4 and O.merkle_fold(real) == bytes(root4.cpu().numpy())
        if world > 1:
            t = torch.tensor([1 if ok4 else 0], device=dev, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok4 = bool(int(t.item()))
        c4 = {"workload": "%d messages x %d rules split over %d GPU(s) (strong scaling), Merkle tree over the scan's event log (32 B / message)" % (C4_MSGS, R, world),
              "msgs_per_s": C4_MSGS / (c4_ms * 1e-3), "ms_per_step": c4_ms, "msgs_this_rank": nc, "scaling": "strong",
              "root_hex": bytes(root4.cpu().numpy()).hex(), "root_equals_oracle": bool(ok4),
              "collective": "all_gather of %d block roots per rank" % nblk4 if world > 1 else "none (1 rank)"}
        del d4, o4, w4, log

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline (oracle port) on a strided sample of the SAME batch, rank 0, N=1 only: every 16th message, so that the
    # comparison of result words covers the whole timed batch, not its first corner
    cpu = None
    if not args.no_cpu and rank == 0 and (world == 1 or os.environ.get("CG_ORACLE_CHECK")):      # (N > 1: only on request, reported as extra.oracle_check)
        from oracle import oracle as O
        regs = [O.Regex(r["source"], "i" if r["flags"] else "") for r in rl]
        threads = host_threads()
        sample = min(int(os.environ.get("CG_CPU_SAMPLE", 65536)), n)
        step_ = max(1, n // sample)
        pick = np.arange(0, sample * step_, step_)
        hb_all = h_data.numpy()[: n * L].reshape(n, L)
        hb = np.concatenate([hb_all[pick].reshape(-1), np.zeros(64, dtype=np.uint8)])
        ho = np.arange(sample + 1, dtype=np.uint64) * L
        warm = min(sample, 2048)
        O.scan_policy(regs, hb[: warm * L + 64], ho[:warm + 1], threads=threads, want_bits=False)
        t0 = time.perf_counter()
        _, cw = O.scan_policy(regs, hb, ho, threads=threads, want_bits=False)
        dt = time.perf_counter() - t0
        agree = bool(np.array_equal(cw, h_words.numpy().view(np.uint64)[pick]))
        cpu = {"value": sample / dt, "unit": "msgs/s", "cores": threads, "per_core": sample / dt / threads, "kind": "port",
               "sample": "every %dth message of the timed batch (%d messages) x %d rules, oracle/jsre.c (-O3; restated oracle, not Node: node %s), %d pinned threads = CPU affinity of the process (os.cpu_count() %s), %.2f s; result words equal to the GPU's: %s"
                         % (step_, sample, R, find_node() or "not found", threads, os.cpu_count(), dt, agree),
               "words_equal_gpu": agree}

    achieved = alg_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms else None
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")     # dram bytes/launch from the committed ncu --set full capture of this kernel
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("scan_kernel_dram_bytes_per_launch")
        except Exception:
            traffic = None
    line = {
        "metric": "messages_scanned_per_s", "value": value, "unit": "msgs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "%d x %dB synthetic msgs x %d-rule firewall scan per GPU (BASELINE configs[1]), policy semantics (RegExp.test per rule), p_hit=%.2f" % (n, L, R, P_HIT),
                   "rules": R, "msg_len": L, "msgs_per_gpu": n, "l2": "inputs (%.0f MB/step) larger than the 126 MB L2" % (n * L / 1e6),
                   "traffic": {"vocabulary_words": args.vocab, "words_sharing_a_prefix_or_suffix_with_a_rule_literal": args.frag_frac, "seed_offset": args.seed_offset,
                               "tuned_on_data": "nothing: the gram filter is compiled from the rule set alone (no profiling pass, no residency)"},
                   "prefilter": {"stride": int(info.stride), "gram_keys": int(info.gram_keys), "level1b_entries": int(info.gram_entries),
                                 "factor_len_min": int(info.factor_len) & 0xff, "factor_len_max": int(info.factor_len) >> 8, "factors": int(info.n_factors),
                                 "bitmap_bytes": int(info.bitmap_bytes), "smem_image_bytes": int(info.image_bytes), "tables_resident": bool(info.tables_resident),
                                 "trigger_bytes": int(info.n_triggers), "always_candidate_rules": int(info.n_always_candidate)},
                   "step": "in-order step replayed as one CUDA graph; results of the timed steps equal the profiled step: %s" % steps_equal,
                   "compile_s": compile_s},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                     "traffic": traffic, "traffic_source": "profiles/traffic.json (dram__bytes_read + write of one ncu --set full capture of this kernel on this workload; not re-measured per run)",
                     "kernel": "scan_kernel", "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": scan_ms, "whole_step_frac": alg_bytes / (ms_per_step * 1e-3) / 1e9 / peak},
        "kernel_ms_note": "kernel_ms: CUDA events inside the library around each kernel of one step (profiling mode, no graph); ms_per_step: the graph-replayed steady state",
        "kernel_ms": {"scan": scan_ms, "confirm": float(kms[1]), "verify": float(kms[2]), "finalize": float(kms[3]),
                      "confirm_parts": {"confirm_kernel": float(kms[4]), "resolve_kernel": float(kms[5])}},
        "candidates": {"flag_words": counters[8], "flagged_grams": counters[6], "grams_past_recheck_map": counters[7], "gram_entry_pairs": counters[9], "confirmed_factor_occurrences": counters[4], "messages_with_candidates": counters[0], "vm_pairs": counters[1], "flags": counters[3],
                       **({"vm_cycle_hist_2^11..": list(counters[8:16]), "vm_cycle_max": counters[7]} if os.environ.get("CG_SCAN_DEBUG") == "2" else {}),
                       "hit_messages": int((words != 0).sum().item()), "injected": len(inj)},
        "cpu_baseline": cpu if world == 1 else None,
        "e2e": {"value": e2e_value, "unit": "msgs/s", "h2d_bytes_per_step": int(n * L + 4 * (n + 1)), "d2h_bytes_per_step": int(8 * n + 64),
                "steps": e2e_steps, "words_equal_device_path": same},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "extra": {"oracle_check": cpu if world > 1 else None, "variants": variants, "merkle": merkle, "c4": c4, "redact": redact, "scan_one": one, "per_rank_ms_per_step": per_rank_ms},
    }
    if args.dump_outputs:
        dump_scan_words(args.dump_outputs, words.cpu().numpy())
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
