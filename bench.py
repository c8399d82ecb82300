#!/usr/bin/env python
"""bench.py — BASELINE config 3: synthetic 2^24-row x 32-column Fp trace ->
iNTT -> coset LDE (blowup 8, bit-reversed rows) -> SHA-256 Merkle commit -> constraint
evaluation over the ce domain, on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps K --warmup W            (N>1: launched by torchrun)
    python bench.py --impl reference ...                     CPU arm: the restated reference CPU
                                                             path (oracle/) on a bounded sample
    python bench.py ... --dump-outputs DIR                   also write a fixed sample of what the
                                                             last timed step computed, as .npy files

Prints ONE JSON line (rank 0).  metric = NTT field-ops/s: the field operations of the step's
transforms (1.5 * N * log2 N per N-point transform, SURVEY.md §8d) divided by the time of the
WHOLE step (transforms + Merkle commit + constraint evaluation), so it moves with "prover
seconds for a 2^24 trace".  See DESIGN.md §Measurement for every key.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N_DEFAULT = 24
NCOLS_DEFAULT = 32
LOG_BLOWUP = 3
L2_BYTES = 126 << 20
DUMP_SAMPLE = 1 << 19       # words kept per dumped array: 3 x (8 MB of halves + 4 MB of indices) stays under 64 MB
DUMP_SEED = 0


def field_ops(log_n, log_b, ncols):
    n, N = 1 << log_n, 1 << (log_n + log_b)
    return ncols * 1.5 * (n * log_n + N * (log_n + log_b))


def algorithmic_bytes(log_n, log_b, ncols):
    """SURVEY.md §8d per phase, 8-byte Fp elements."""
    n, N = 1 << log_n, 1 << (log_n + log_b)
    return {
        "intt": 2 * 8 * n * ncols,
        "lde": (8 * n + 8 * N) * ncols,
        "leaf_hash": (8 * ncols + 32) * N,
        "merkle_nodes": 96 * (N - 1),
        "constraint_eval": ((ncols + 1) * 8 + 8) * n,
    }


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 7:
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(self.rows), "reasons": sorted(reasons)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """per-launch DRAM bytes of the dominant kernel from the committed ncu summary, or None"""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return None


def golden_entry(log_n, ncols, world):
    """committed oracle outputs for this workload (tests/golden/config3.json, made by tests/golden/make_config3_golden.py):
    the bench never runs the oracle for this — it compares against the fixture"""
    p = os.path.join(ROOT, "tests", "golden", "config3.json")
    try:
        return json.load(open(p)).get(f"2^{log_n}x{ncols}x{world}")
    except Exception:
        return None


def check_against_golden(g, root, ce_tensor, what):
    import hashlib
    if g is None:
        return {"golden": None, "note": f"no committed fixture for {what}"}
    got_root = root.hex()
    ce_sha = hashlib.sha256(ce_tensor.cpu().numpy().tobytes()).hexdigest()
    ok_root, ok_ce = got_root == g["merkle_root"], ce_sha == g["constraint_eval_sha256"]
    if not (ok_root and ok_ce):
        raise SystemExit(f"bench: {what}: result differs from the oracle fixture: root {got_root} vs {g['merkle_root']}, "
                         f"constraint column sha256 {ce_sha} vs {g['constraint_eval_sha256']}")
    return {"golden": "tests/golden/config3.json", "case": what, "merkle_root": True, "constraint_eval_sha256": True}


def dump_outputs(out_dir, root, arrays):
    """Writes a step's outputs to out_dir as float64 .npy files, so that two builds can be compared output for output:
    merkle_root.npy holds the root's 32 bytes; for every device array of 64-bit field words (Montgomery form, as the
    library returns them), <name>.npy holds a sample of shape (k, 2), the low and high 32-bit halves of each word (exact
    in float64), and <name>_index.npy the flat row-major index of each sampled word.  The sample is the whole array up to
    DUMP_SAMPLE words, else DUMP_SAMPLE positions drawn with a fixed seed: it depends only on the array's size."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "merkle_root.npy"), np.frombuffer(root, dtype=np.uint8).astype(np.float64))
    for name, t in arrays.items():
        flat = t.reshape(-1)
        total = flat.numel()
        if total <= DUMP_SAMPLE:
            idx = np.arange(total, dtype=np.int64)
        else:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(total, DUMP_SAMPLE, replace=False))
        words = np.ascontiguousarray(flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy())
        np.save(os.path.join(out_dir, f"{name}.npy"), words.view("<u4").reshape(-1, 2).astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))


# ----------------------------------------------------------------------------- CPU arm
def cpu_sample(log_n, ncols, log_b, steps=1):
    """The restated reference CPU path (oracle/gl_oracle.c, all host threads) on a bounded sample:
    same pipeline, 2^log_n rows.  Returns (seconds per step, field-ops/s, threads, root)."""
    from oracle import oracle as orc
    from oracle import synth_oracle
    threads = pick_cpu_threads(orc, synth_oracle, ncols, log_b)
    trace = orc.rand_matrix(ncols, 1 << log_n, 1, seed=3000)
    best = None
    root = None
    for _ in range(steps):
        t0 = time.perf_counter()
        polys = orc.ntt(trace, 1, log_n, inverse=True)
        lde = orc.lde(polys, 1, log_n, log_b, orc.generator(), bitrev=True)
        nodes = orc.merkle_nodes(orc.hash_rows(lde, 1))
        synth_oracle.constraint_eval(orc, lde, log_n, log_b, ncols)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
        root = nodes[1].tobytes()
    return best, field_ops(log_n, log_b, ncols) / best, threads, root


_CPU_THREADS = None


def pick_cpu_threads(orc, synth_oracle, ncols, log_b):
    """Give the CPU arm its best thread count: OpenMP's default (all logical CPUs) can oversubscribe a
    cgroup-limited or hyper-threaded host badly, so a tiny instance of the pipeline is timed at a few
    candidate counts (logical CPUs available to this process, half, quarter) and the fastest is kept."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        orc.lib().orc_set_num_threads(_CPU_THREADS)
        return _CPU_THREADS
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cands = sorted({max(1, avail), max(1, avail // 2), max(1, avail // 4)}, reverse=True)
    log_n = 14
    trace = orc.rand_matrix(ncols, 1 << log_n, 1, seed=1)
    best = None
    for t in cands:
        orc.lib().orc_set_num_threads(t)
        dt = None
        for _ in range(2):
            t0 = time.perf_counter()
            polys = orc.ntt(trace, 1, log_n, inverse=True)
            lde = orc.lde(polys, 1, log_n, log_b, orc.generator(), bitrev=True)
            orc.merkle_nodes(orc.hash_rows(lde, 1))
            synth_oracle.constraint_eval(orc, lde, log_n, log_b, ncols)
            d = time.perf_counter() - t0
            dt = d if dt is None else min(dt, d)
        if best is None or dt < best[0]:
            best = (dt, t)
    _CPU_THREADS = best[1]
    orc.lib().orc_set_num_threads(_CPU_THREADS)
    return _CPU_THREADS


def full_prove_sample(log_rows=21):
    """the whole default_prove on the reference's own example (examples/fib at its native size, main.rs:225-229):
    host trace -> proof object, checked by the restated verifier (the oracle as checker, not as the thing measured)"""
    import time
    from ministark_b200.air import Air, ProofOptions
    from ministark_b200.examples import fib
    from ministark_b200.prover import GpuProver
    from oracle import stark_oracle
    trace, last = fib.gen_trace(8 << log_rows, pinned=True)      # page-locked columns, like the reference's GpuAllocator
    claim = fib.FibClaim(last)
    prover = GpuProver(0)
    prover.prove(claim, fib.OPTIONS, trace)
    best = None
    for _ in range(3):
        t = time.perf_counter()
        proof = prover.prove(claim, fib.OPTIONS, trace)
        dt = time.perf_counter() - t
        best = (dt, proof) if best is None or dt < best[0] else best
    dt, proof = best
    pb = proof.to_bytes()
    stark_oracle.verify(claim, pb, fib.SECURITY_LEVEL, lambda n, o: Air(claim.AirConfig, n, claim.get_public_inputs(), ProofOptions(*o)))
    return {"workload": f"examples/fib: 2^{log_rows} rows x 8 Fp columns, ProofOptions(32, 4, 8, 8, 64), pinned host trace -> proof",
            "seconds": dt, "phases_s": {k: round(v, 5) for k, v in proof.timings.items()}, "proof_bytes": len(pb),
            "verified": True, "launches": prover.ctx.launches}


def cpu_full_prove_sample(log_rows):
    """default_prove in the reference's own formulation on the host cores (oracle/stark_oracle.cpu_prove: per-column
    transforms, coefficient-form DEEP, apply_drp through two transforms, CPU Merkle), examples/fib, checked by the
    restated verifier — the CPU counterpart of full_prove_sample at a size that stays within the time budget"""
    import time
    from ministark_b200.air import Air, ProofOptions
    from ministark_b200.examples import fib
    from oracle import stark_oracle
    trace, last = fib.gen_trace(8 << log_rows)
    claim = fib.FibClaim(last)
    mk = lambda n, o: Air(claim.AirConfig, n, claim.get_public_inputs(), ProofOptions(*o))
    t = time.perf_counter()
    proof = stark_oracle.cpu_prove(claim, (32, 4, 8, 8, 64), trace.base_columns(), mk)
    dt = time.perf_counter() - t
    stark_oracle.verify(claim, proof, fib.SECURITY_LEVEL, mk)
    return {"workload": f"examples/fib: 2^{log_rows} rows x 8 Fp columns, ProofOptions(32, 4, 8, 8, 64), CPU restatement of default_prove",
            "seconds": dt, "proof_bytes": len(proof), "verified": True}


def cpu_full_prove_compiled(log_rows):
    """the C++ default_prove (include/ministark_prover.hpp) linked against the CPU build of the C ABI (oracle/cpu_abi.c):
    a prover compiled end to end on the host cores — same formulation as the GPU driver (kind "port"), proof bytes
    identical to cpu_prove's (tests/test_cpp_cpu_abi.py), checked by the C++ verifier inside the binary"""
    odir = os.path.join(ROOT, "oracle")
    exe = os.path.join(odir, "cpu_prover")
    try:
        subprocess.check_call(["make", "-s", "-C", odir, "cpu_prover"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        out = subprocess.run([exe, str(log_rows), "32", "4", "8", "8", "64"], capture_output=True, text=True, timeout=1800)
        if out.returncode != 0:
            return {"unavailable": out.stderr.strip()[-200:]}
        r = json.loads(out.stdout)
    except Exception as e:      # no compiler / no binary: the Python-orchestrated sample above still stands
        return {"unavailable": repr(e)[:200]}
    return {"workload": f"examples/fib: 2^{log_rows} rows x 8 Fp columns, ProofOptions(32, 4, 8, 8, 64), C++ default_prove on the CPU "
                        "build of the C ABI (evaluation-form DEEP, per-coset FRI fold: the GPU driver's formulation)",
            "seconds": r["seconds"], "proof_bytes": r["proof_bytes"], "verified": r["verified"], "cores": r["threads"], "kind": "port"}


def cpu_brainfuck_prove_compiled(burner):
    """examples/brainfuck, program cycle_burner(a, b, c) (40,40,60: 2^20 rows — the size of the GPU figure in
    profiles/bench_brainfuck_burner_*.json), ProofOptions(19, 16, 20, 16, 16), through the same compiled CPU prover"""
    from ministark_b200.examples import brainfuck as bf
    odir = os.path.join(ROOT, "oracle")
    try:
        a, b, c = (int(v) for v in burner.split(","))
        ii, mi = bf.test_rng_fq3(2)
        subprocess.check_call(["make", "-s", "-C", odir, "cpu_prover"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        out = subprocess.run([os.path.join(odir, "cpu_prover"), "bf", str(a), str(b), str(c), "19", "16", "20", "16", "16"] + [str(v) for v in ii + mi],
                             capture_output=True, text=True, timeout=3600)
        if out.returncode != 0:
            return {"unavailable": out.stderr.strip()[-200:]}
        r = json.loads(out.stdout)
    except Exception as e:
        return {"unavailable": repr(e)[:200]}
    return {"workload": f"examples/brainfuck: cycle_burner({a},{b},{c}), {r['rows']} rows x (17 Fp + 9 Fq3) columns, ProofOptions(19, 16, 20, 16, 16), "
                        "C++ default_prove on the CPU build of the C ABI (VM run excluded)",
            "seconds": r["seconds"], "proof_bytes": r["proof_bytes"], "verified": r["verified"], "cores": r["threads"], "kind": "port"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    log_n = args.cpu_log_n
    no_prover = args.no_prover or args.gpus > 1
    t0 = time.perf_counter()
    for _ in range(args.warmup and 1):
        cpu_sample(log_n, args.ncols, LOG_BLOWUP)
    times = []
    val = 0.0
    threads = 1
    for _ in range(args.steps):
        dt, val_i, threads, _ = cpu_sample(log_n, args.ncols, LOG_BLOWUP)
        times.append(dt)
    ms = 1000 * sum(times) / len(times)
    val = field_ops(log_n, LOG_BLOWUP, args.ncols) / (ms / 1000)
    sample = (f"2^{log_n}-row x {args.ncols}-col trace (1/{1 << (args.log_n - log_n)} of the rows), all phases, "
              f"{threads} host threads, oracle/gl_oracle.c restated reference CPU path")
    print(json.dumps({
        "impl": "reference", "metric": "ntt_field_ops_per_s", "value": val, "unit": "field-ops/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": "field-ops/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "field-ops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "timed_sample": {"rows_log2": log_n, "of_rows_log2": args.log_n,
                         "note": "the CPU arm times this bounded sample of the workload; the metric is throughput, normalised by the "
                                 "field operations of the sample"},
        # CPU proves of the GPU arm's full-prove workloads (N-independent: reported with the N = 1 line only)
        "full_prove": None if no_prover else cpu_full_prove_sample(args.cpu_prove_log_rows),
        "full_prove_compiled": None if no_prover else cpu_full_prove_compiled(args.cpu_prove_log_rows),
        "brainfuck_prove_compiled": None if no_prover or not args.cpu_bf_burner else cpu_brainfuck_prove_compiled(args.cpu_bf_burner),
        "wall_s": time.perf_counter() - t0,
    }))


def workload_config(args):
    total_cols = args.ncols * (args.gpus if args.impl != "reference" else 1)
    shape = (f"2^{args.log_n}-row x {args.ncols}-col" if args.gpus == 1 or args.impl == "reference" else
             f"2^{args.log_n}-row x {total_cols}-col ({args.ncols} columns per GPU: weak scaling)")
    # (both arms print the SAME config: the reference arm states the size of the sample it times in `timed_sample`
    #  and in cpu_baseline.sample, outside this dict)
    return {"workload": f"config3: synthetic {shape} Fp trace, iNTT + coset LDE x{1 << LOG_BLOWUP} "
                        "(bit-reversed) + SHA-256 Merkle commit + constraint eval (32 degree-2 transition constraints per "
                        "32-column block, ce_blowup 1)",
            "log_n": args.log_n, "ncols": total_cols, "ncols_per_gpu": args.ncols, "blowup": 1 << LOG_BLOWUP,
            "l2_policy": "inputs (>= 4 GiB per phase) far exceed the 126 MB L2; no explicit flush",
            "parallelism": ("single GPU" if args.gpus == 1 else
                            f"{args.gpus} ranks: one {args.ncols * args.gpus}-column trace, {args.ncols}-column block per rank "
                            "(iNTT/LDE local), " +
                            ("LDE then NCCL all-to-all into row slabs" if args.no_fused_exchange else
                             "LDE whose last pass stores each coset block into the owner's row slab over NVLink (CUDA IPC peer "
                             "memory; no all-to-all)") +
                            " for the leaf hash, all-gather of subtree roots and of the partial composition sums")}


# ----------------------------------------------------------------------------- verification and extra arms
def sharded_small_check(ctx, dist, dev, stream, world, rank, args):
    """N > 1: the sharded commit + partial-composition path of the timed step, on a 2^16-row x 32*N-column instance whose
    root and constraint column are committed oracle outputs (tests/golden/config3.json)"""
    import torch

    import ministark_b200 as ms
    from ministark_b200 import parallel, synth_air
    log_n, log_b, ncols = 16, LOG_BLOWUP, 32
    g = golden_entry(log_n, ncols, world)
    n = 1 << log_n
    tr = torch.empty((ncols, n), dtype=torch.int64, device=dev)
    ctx.fill_random(tr, ncols * n, 3000 + rank)
    sc = parallel.ShardedCommit(parallel.CudaEngine(ctx, dev, stream=stream), dist, log_n, log_b, ncols * world,
                                fused=False if args.no_fused_exchange else None)
    sc.transform(tr)
    root = sc.commit()
    ev = synth_air.GpuConstraintEval(ctx, log_n, log_b, ncols, dev)
    ce = torch.empty(n, dtype=torch.int64, device=dev)
    ev.run(sc.lde, ce)
    parts = torch.empty((world, n), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(parts, ce)
    ctx.sum_columns(parts, ce, ms.FP, n, world)
    ctx.sync()
    out = check_against_golden(g, root, ce, f"2^{log_n} x {ncols * world} over {world} GPUs (fused exchange: {sc.fused})")
    sc.close()
    return out


class _FriChannel:
    """stands in for fri::ProverChannel (src/channel.rs:122-140) in the config-4 sweep: fixed alphas, roots recorded"""

    def __init__(self):
        self.roots, self.k = [], 0

    def commit_fri_layer(self, root):
        self.roots.append(root)

    def draw_fri_alpha(self):
        self.k += 1
        return (3 + self.k, 5, 7)


def _fri_single(prover, cur, log_n, fq, options, channel):
    """FriProver::build_layers on one GPU (the loop of ministark_b200/prover.py)"""
    import numpy as np
    ctx = prover.ctx
    ff = options.fri_folding_factor
    log_ff = ff.bit_length() - 1
    ln = log_n
    for _ in range(options.fri_num_layers(1 << log_n)):
        nrows = 1 << (ln - log_ff)
        leaves, nodes = prover._empty(nrows, 4), prover._empty(nrows, 4)
        channel.commit_fri_layer(ctx.merkle_commit_rows(cur, ff * fq, nrows, leaves=leaves, nodes=nodes))
        alpha = channel.draw_fri_alpha()
        nxt = prover._empty(nrows * fq)
        ctx.fri_fold(cur, nxt, fq, ln, log_ff, np.array([c * 2**64 % (2**64 - 2**32 + 1) for c in alpha], dtype=np.uint64))
        cur, ln = nxt, ln - log_ff
    return cur


def extra_arms(args, dist, dev, world, rank):
    """(1) strong scaling: the FIXED 2^24 x 32 workload over N GPUs, every matrix sharded by LDE coset blocks
    (ministark_b200/prover_mgpu.py), root and constraint column checked against the full-size oracle fixture;
    (2) BASELINE config 4: FRI commit phase (every layer: row hashes, tree, fold) of Fq3 codewords 2^20..2^26 on N GPUs;
    (3) BASELINE config 5 (fib substitute, SURVEY 8d): the whole default_prove of a 2^22-row trace on N GPUs."""
    import hashlib

    import numpy as np
    import torch

    import ministark_b200 as ms
    from ministark_b200 import synth_air
    from ministark_b200.air import Air, ProofOptions
    from ministark_b200.examples import fib
    from ministark_b200.prover import GpuProver
    if dist is not None:
        from ministark_b200.prover_mgpu import ShardedProver
        sp = ShardedProver(dist, dev.index)
    else:
        sp = GpuProver(dev.index)
    ctx = sp.ctx

    def timed(fn, reps):
        fn()
        best = None
        for _ in range(reps):
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            best = (float(t.item()), out) if best is None or float(t.item()) < best[0] else best
        return best

    strong = fri = prove = None
    with torch.cuda.stream(sp.stream):
        # ---- (1) strong scaling
        log_n, log_b, ncols = args.log_n, LOG_BLOWUP, args.ncols
        if dist is not None and (1 << log_b) % world == 0 and ncols % world == 0:
            n, N = 1 << log_n, 1 << (log_n + log_b)
            rows_per = N // world
            full = sp._empty(ncols, n)
            ctx.fill_random(full, ncols * n, 3000)            # the N = 1 workload; every rank holds the host-side trace
            prog = synth_air.GpuConstraintEval(ctx, log_n, log_b, ncols, dev).prog
            ce = sp._empty(n)

            def strong_step():
                polys = sp._interpolate(full, ms.FP, ncols, log_n)            # 1/N of the columns each + all-gather
                slab = sp._lde_slab(polys, ms.FP, ncols, log_n, log_b)        # this rank's coset blocks of every column
                _, root = sp._commit_slab(slab, ms.FP, ncols, rows_per)       # subtree + all-gather of the roots
                if rank == 0:                                                  # ce_blowup 1: the ce domain is block 0
                    ctx.eval_constraints_ptrs(prog, ce, log_n, sp._block_ptrs(slab, ms.FP, ncols, rows_per, 0, n),
                                              [False] * ncols, fq_field=ms.FP, offset=ms.GENERATOR, trace_bitrev=True)
                dist.broadcast(ce, src=0)
                return root

            ms_step, root = timed(strong_step, max(1, min(args.steps, 5)))
            ver = None if args.no_verify else check_against_golden(
                golden_entry(log_n, ncols, 1), root, ce, f"2^{log_n} x {ncols} over {world} GPUs (strong scaling)")
            strong = {"workload": f"the N = 1 workload unchanged (2^{log_n} x {ncols}, blow-up {1 << log_b}) over {world} GPUs: iNTT of "
                                  f"{ncols // world} columns per rank, NCCL all-gather of the coefficients, LDE + leaf hashes + subtree of "
                                  f"{(1 << log_b) // world} coset block(s) of every column per rank, all-gather of subtree roots, "
                                  "constraint evaluation on the rank that owns the ce block + broadcast",
                      "ms_per_step": ms_step, "value": field_ops(log_n, log_b, ncols) / (ms_step / 1000), "unit": "field-ops/s",
                      "verified": ver}
            del full, ce
            torch.cuda.empty_cache()

        # ---- (2) config 4: FRI commit phase of Fq3 codewords
        fri = []
        opts = ProofOptions(32, 8, 0, 8, 64)
        for lg in (20, 22, 24, 26):
            words = 3 * (1 << lg) // world
            slab = sp._empty(words)
            ctx.fill_random(slab, words, 4000 + 16 * lg + rank)

            def fri_step():
                ch = _FriChannel()
                if dist is not None:
                    sp.fri_commit(slab, lg, ms.FQ3, opts, ch)
                else:
                    _fri_single(sp, slab, lg, ms.FQ3, opts, ch)
                return ch.roots

            t_ms, roots = timed(fri_step, 3)
            rec = {"log_n": lg, "field": "Fq3", "ff": 8, "layers": len(roots), "gpus": world, "ms": t_ms,
                   "GBps_algorithmic": (24 * (1 << lg) * (1 + 1 / 8)) / (t_ms / 1000) / 1e9, "layer0_root": roots[0].hex()}
            if dist is not None:                  # the same codeword through the single-GPU loop on rank 0: same roots
                full = sp._empty(3 * (1 << lg))
                dist.all_gather_into_tensor(full, slab)
                if rank == 0:
                    ch = _FriChannel()
                    _fri_single(sp, full, lg, ms.FQ3, opts, ch)
                    if ch.roots != roots:
                        raise SystemExit(f"bench: sharded FRI roots differ from the single-GPU roots at 2^{lg}")
                    rec["roots_equal_single_gpu"] = True
                del full
            fri.append(rec)
            del slab
            torch.cuda.empty_cache()

    # ---- (3) config 5: the whole prover on a 2^22-row examples/fib trace
    if not args.no_prover and (dist is None or 8 % world == 0):
        import time
        log_rows, o5 = args.prove_log_rows, (32, 8, 8, 8, 64)
        trace, last = fib.gen_trace(8 << log_rows, pinned=True)     # page-locked columns, like the reference's GpuAllocator
        claim = fib.FibClaim(last)
        options = ProofOptions(*o5)
        sp.prove(claim, options, trace)
        best = None
        for _ in range(3):
            if dist is not None:
                dist.barrier()
            t0 = time.perf_counter()
            proof = sp.prove(claim, options, trace)
            dt = torch.tensor([time.perf_counter() - t0], device=dev)
            if dist is not None:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            best = (float(dt.item()), proof) if best is None or float(dt.item()) < best[0] else best
        dt, proof = best
        pb = proof.to_bytes()
        digest = hashlib.sha256(pb).hexdigest()
        if dist is not None:
            all_d = [None] * world
            dist.all_gather_object(all_d, digest)
            if len(set(all_d)) != 1:
                raise SystemExit("bench: ranks disagree on the proof bytes")
        if rank == 0:
            from oracle import stark_oracle       # the restated verifier as CHECKER of the timed proof, outside the timed region
            stark_oracle.verify(claim, pb, 20, lambda nn, oo: Air(claim.AirConfig, nn, claim.get_public_inputs(), ProofOptions(*oo)))
        prove = {"workload": f"examples/fib: 2^{log_rows} rows x 8 Fp columns, ProofOptions{o5} (blow-up 8 so that the 8 coset "
                             "blocks shard over up to 8 GPUs; the reference example uses blow-up 4), host trace -> proof bytes",
                 "gpus": world, "seconds": dt, "phases_s": {k: round(v, 5) for k, v in proof.timings.items()},
                 "proof_bytes": len(pb), "proof_sha256": digest, "verified": True}
    return strong, fri, prove


# ----------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist

    import ministark_b200 as ms
    from ministark_b200 import synth_air

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    log_n, log_b, ncols = args.log_n, LOG_BLOWUP, args.ncols
    n, N = 1 << log_n, 1 << (log_n + log_b)
    # a dedicated (non-default) torch stream: the library launches on it, torch events time on it
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)
    ctx = ms.Context(local, stream=stream.cuda_stream)

    dev = torch.device("cuda", local)
    from ministark_b200.pipeline import TraceCommitPipeline
    evaluator = synth_air.GpuConstraintEval(ctx, log_n, log_b, ncols, dev)
    pipe = TraceCommitPipeline(ctx, dev, log_n, log_b, ncols, evaluator=evaluator, chunk_cols=4, stream=stream)
    trace, polys, lde, ce_out = pipe.trace, pipe.polys, pipe.lde, pipe.ce
    ctx.fill_random(trace, ncols * n, 3000 + rank)
    host_trace = None
    sharded = partials = None
    if world > 1:
        # one trace of ncols*world columns, column blocks sharded over the ranks (ministark_b200/parallel.py):
        # local iNTT + LDE, all-to-all into row slabs, slab hash + subtree, all-gather of the subtree roots;
        # the composition is a sum over column-local constraint groups: partial sums are all-gathered and added
        from ministark_b200 import parallel
        sharded = parallel.ShardedCommit(parallel.CudaEngine(ctx, dev, stream=stream), dist, log_n, log_b, ncols * world,
                                         polys=polys, lde=lde, fused=False if args.no_fused_exchange else None)
        if sharded.fused:
            pipe.lde_fn = sharded.lde_columns
        partials = torch.empty((world, n), dtype=torch.int64, device=dev)

    def commit():
        return sharded.commit() if sharded is not None else pipe.commit()

    def evaluate():
        pipe.evaluate()
        if sharded is not None:
            dist.all_gather_into_tensor(partials, ce_out)
            ctx.sum_columns(partials, ce_out, ms.FP, n, world)

    def step():
        """device-resident step, phase by phase (the same calls TraceCommitPipeline.run_resident makes)"""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        if sharded is not None and sharded.fused:
            # the last LDE pass stores its blocks into the owners' row slabs over NVLink: that pass is link-bound, the
            # others ALU-bound, so the columns go through in chunks — chunk k's store-heavy pass overlaps the peers'
            # arithmetic of chunk k +- 1 instead of every rank hitting the links at once (SCALE_r01: the chunked
            # end-to-end path beat the monolithic resident step at N >= 4)
            ev[1].record()
            for c0 in range(0, ncols, pipe.chunk):
                k = min(pipe.chunk, ncols - c0)
                ctx.ntt_batch_to(trace[c0], polys[c0], ms.FP, log_n, k, inverse=True)
                sharded.lde_columns(c0, k)
        else:
            ctx.ntt_batch_to(trace, polys, ms.FP, log_n, ncols, inverse=True)
            ev[1].record()
            ctx.lde_batch(polys, lde, ms.FP, log_n, log_b, ncols, offset=ms.GENERATOR, bitrev=True)
        ev[2].record()
        root = commit()                                                                # D2H of the 32-byte root
        ev[3].record()
        evaluate()
        ev[4].record()
        return ev, root

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value)
    for _ in range(args.warmup):
        step()
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    l0 = ctx.launches
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    evs = []
    root = None
    for _ in range(args.steps):
        e, root = step()
        evs.append(e)
    t_end.record()
    barrier()
    launches = ctx.launches - l0
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        # the last timed step's results, before the end-to-end steps below recompute them into the same buffers
        arrays = {"constraint_eval": ce_out}
        if world == 1:      # at N > 1 polys holds this rank's column block and lde the exchange's work buffer
            arrays.update(polys=polys, lde=lde)
        dump_outputs(args.dump_outputs, root, arrays)
    total_ms = t_start.elapsed_time(t_end)
    names = ["intt", "lde", "merkle", "constraint_eval"]
    phase_ms = {nm: sum(e[i].elapsed_time(e[i + 1]) for e in evs) / args.steps for i, nm in enumerate(names)}
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    ops = field_ops(log_n, log_b, ncols) * world
    value = ops / (ms_per_step / 1000)

    # ---- end to end through the public API (TraceCommitPipeline.run_from_host) with HOST buffers: pinned
    #      host trace -> chunked H2D overlapped with iNTT/LDE -> Merkle commit -> constraint evaluation
    #      -> D2H of the root and of the composition-evaluation column
    if args.no_e2e:     # profiling runs (profiles/capture.sh): resident steps only
        if rank == 0:
            print(json.dumps({"note": "resident steps only (--no-e2e)", "ms_per_step": ms_per_step, "phase_ms": phase_ms}))
        if world > 1:
            dist.destroy_process_group()
        return
    host_trace = torch.empty((ncols, n), dtype=torch.int64, pin_memory=True)
    host_trace.copy_(trace)
    e2e_steps = max(1, min(args.steps, 3))
    host_ce = torch.empty(n, dtype=torch.int64, pin_memory=True)

    def e2e_step():
        return pipe.run_from_host(host_trace, commit_fn=commit, evaluate_fn=evaluate)[0]

    e2e_step()
    barrier()
    t_start.record()
    e2e_root = None
    for _ in range(e2e_steps):
        e2e_root = e2e_step()
    t_end.record()
    barrier()
    assert e2e_root == root, "e2e path and resident path disagree on the Merkle root"
    e2e_ms = t_start.elapsed_time(t_end) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = ops / (e2e_ms / 1000)

    # ---- the timed result against the committed oracle fixture: at N = 1 the full-size root and the digest of the
    #      constraint-evaluation column; at N > 1 the same sharded code path on a 2^16-row instance (fixtures exist for
    #      32 * N columns, N = 2, 4, 8) — the full-size multi-GPU check is the strong-scaling arm below
    verified = None
    if not args.no_verify:
        if world == 1:
            verified = check_against_golden(golden_entry(log_n, ncols, 1), root, ce_out, f"2^{log_n} x {ncols}, 1 GPU")
        else:
            verified = sharded_small_check(ctx, dist, dev, stream, world, rank, args)
    strong = fri = sharded_prove = None
    if world > 1 and not args.no_extra:
        # free the weak-scaling buffers first: the arms below allocate their own
        del pipe, evaluator, trace, polys, lde, ce_out, partials, host_trace, host_ce
        sharded.close()
        del sharded
        torch.cuda.empty_cache()
    if not args.no_extra:
        strong, fri, sharded_prove = extra_arms(args, dist if world > 1 else None, dev, world, rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel family (the NTT pass kernels: msntt::ntt_tma_kernel, the persistent TMA
    #      pipeline): the LDE is 3 launches of it; achieved = algorithmic LDE bytes / device time of those launches
    #      (CUDA events on the launching stream); raw = the DRAM bytes ncu counted for the same launches / the same time.
    alg = algorithmic_bytes(log_n, log_b, ncols)
    peak, peak_src = measured_peak_hbm()
    lde_gbs = alg["lde"] / (phase_ms["lde"] / 1000) / 1e9
    traffic = ncu_traffic()
    raw = None
    if traffic and traffic.get("lde_dram_bytes_per_launch") and world == 1:
        raw_gbs = 3 * traffic["lde_dram_bytes_per_launch"] / (phase_ms["lde"] / 1000) / 1e9
        raw = {"achieved": raw_gbs, "frac": raw_gbs / peak, "unit": "GB/s",
               "note": "ncu dram__bytes (read + write) of the 3 LDE launches / their CUDA-event time: each of the three 8-bit "
                       "passes streams the whole 32 GiB once (the north-star's >= 60 % target is on this figure)"}
    roofline = {"kernel": "msntt::ntt_tma_kernel (LDE: 3 launches of the persistent TMA pipeline)", "bound": "hbm",
                "achieved": lde_gbs, "peak": peak,
                "unit": "GB/s", "frac": lde_gbs / peak, "peak_source": peak_src,
                "traffic": traffic.get("lde_dram_bytes_per_launch") if traffic else None, "raw_dram": raw,
                "algorithmic_bytes": alg["lde"], "launch_ms_sum": phase_ms["lde"],
                "per_phase_GBps": {k: (alg[k2] / (phase_ms[k] / 1000) / 1e9) for k, k2 in
                                   (("intt", "intt"), ("lde", "lde"), ("constraint_eval", "constraint_eval"))},
                "merkle_GBps": (alg["leaf_hash"] + alg["merkle_nodes"]) / (phase_ms["merkle"] / 1000) / 1e9,
                "ncu_pipe_utilisation": traffic.get("ncu_pipe_utilisation") if traffic else None,
                "note": "integer-ALU bound (64-bit modular arithmetic on 32-bit lanes: ALU pipe 71-85 % busy, DESIGN.md 5.1): the "
                        "algorithmic HBM fraction is low by construction; raw_dram is the figure comparable with a streaming kernel"}

    # ---- CPU baseline: restated reference CPU path on a bounded sample, host cores of this box
    cpu = None
    if not args.no_cpu and world == 1:      # the CPU baseline is a rank-0, N = 1 measurement
        dt, cval, threads, _ = cpu_sample(args.cpu_log_n, ncols, log_b)
        cpu = {"value": cval, "unit": "field-ops/s", "cores": threads, "kind": "port", "seconds": dt,
               "sample": f"2^{args.cpu_log_n}-row x {ncols}-col trace (1/{1 << (log_n - args.cpu_log_n)} of the rows), all phases, "
                         "oracle/gl_oracle.c (restated reference CPU path, OpenMP over all host threads)"}

    full_prove = None
    if world == 1 and not args.no_e2e and not args.no_prover:
        full_prove = full_prove_sample()      # ~2 GiB next to the resident config-3 buffers

    out = {
        "metric": "ntt_field_ops_per_s", "value": value, "unit": "field-ops/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config(args),
        "step_s": ms_per_step / 1000, "phase_ms": phase_ms, "gpu_launches": launches, "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "field-ops/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": ncols * n * 8, "d2h_bytes_per_step": 32 + n * 8},
        "roofline": roofline, "cpu_baseline": cpu, "merkle_root": root.hex() if root else None,
        "verified": verified, "full_prove": full_prove,
        "strong_scaling": strong, "config4_fri": fri, "config5_sharded_prove": sharded_prove,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=LOG_N_DEFAULT)
    ap.add_argument("--ncols", type=int, default=NCOLS_DEFAULT)
    ap.add_argument("--cpu-log-n", type=int, default=20, help="rows of the bounded CPU sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="resident steps only (for ncu captures)")
    ap.add_argument("--no-prover", action="store_true", help="skip the examples/fib full-prove sample")
    ap.add_argument("--prove-log-rows", type=int, default=22, help="rows of the config-5 (sharded) full-prove sample")
    ap.add_argument("--cpu-bf-burner", default="40,40,60", help="--impl reference: cycle_burner(a,b,c) of the compiled CPU brainfuck prove "
                    "(40,40,60 = 2^20 rows; empty string: skip)")
    ap.add_argument("--cpu-prove-log-rows", type=int, default=21, help="--impl reference: rows of the CPU full-prove sample")
    ap.add_argument("--no-fused-exchange", action="store_true", help="N > 1: LDE then NCCL all-to-all instead of the fused scatter")
    ap.add_argument("--no-verify", action="store_true", help="skip the comparison with the committed oracle fixtures")
    ap.add_argument("--no-extra", action="store_true", help="skip the strong-scaling, FRI-sweep and sharded-prover arms")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                    "(float64; the Merkle root, the constraint column and, at N = 1, the coefficients and the LDE, each "
                    "sampled at fixed positions to at most 2^19 words)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm's timed step")
    args.cpu_log_n = min(args.cpu_log_n, args.log_n)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
