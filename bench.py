#!/usr/bin/env python
"""bench.py — step ready-evaluations/sec of the StoryRun DAG frontier pass.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config 3] [--dump-outputs DIR]

A "step" is one frontier pass over one batch of synthetic StoryRuns: BASELINE.json
configs[2] — 100k StoryRuns x 256 steps, random DAG with in-degree 4 — per GPU (weak
scaling: every rank evaluates its own 100k-run shard; the only cross-GPU traffic is one
NCCL all-gather of the per-shard counts per pass).  One evaluation = one (StoryRun, step)
visit of the findReadySteps loop (dag.go:2647).

Prints ONE JSON line (rank 0).  `value` = device-timed throughput with inputs resident in
HBM; `e2e` = the same metric through the public host-buffer calls (pinned host buffers,
H2D + kernels + D2H inside the timed region); `roofline` relates the kernel's algorithmic
bytes to the measured HBM copy peak; `cpu_baseline` times the CPU oracle on the box's host
cores (a reported baseline, not the target); `configs` carries the other BASELINE.json
configurations (cfg4 at every N, cfg5 = 125k runs x 1024 steps per GPU, 1M x 1024 at 8
GPUs) and `parity_check` the byte-for-byte comparison of the FULL benchmarked batches with
the oracle (outside the timed regions; the line is withheld and the exit code non-zero when
it fails).

Timing protocol: the K-step region is one or more CUDA-graph replays whose unroll divides K
(no eager tail), it starts right after a device-side rendezvous (a one-element all-reduce on
the launching stream) so every rank's region starts aligned, and it is repeated `--reps`
times; each repetition is bracketed by CUDA events, reduced with MAX over ranks, and the
MEDIAN repetition is reported (all of them are listed in `timing.region_ms`).

--impl reference times the reference's algorithm on the CPU.  The reference is Go and there
is no Go toolchain in this image (nor network), so the CPU arm is the oracle restatement
(kind "port") on bounded samples of the same workload.  That arm never loads the CUDA library.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "step ready-evals/sec @100k StoryRuns x 256 steps"
UNIT = "evals/s"

# bits of the header constants the CPU arm needs (it must not load the CUDA library; tests check them against _abi)
F_COND, F_DECISION, F_CHILD = 0x1, 0x2, 0x4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60, help="frontier passes in each timed repetition (see --reps)")
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, help="BASELINE.json config index (2..5), default 3 = configs[2]")
    ap.add_argument("--runs", type=int, default=0, help="StoryRuns per GPU (default: the config's N, 125k for cfg 5)")
    ap.add_argument("--rot", type=int, default=3, help="disjoint input copies rotated between passes (L2 hygiene)")
    ap.add_argument("--reps", type=int, default=11, help="repetitions of the K-step timed region (median reported)")
    ap.add_argument("--cpu-sample-runs", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg4 / cfg5 legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-size comparison with the oracle")
    ap.add_argument("--shared", type=int, default=0, help="shared-topology mode: D distinct topologies (0 = unique)")
    ap.add_argument("--ncu", action="store_true", help="profiling run: few eager passes, no e2e / cpu / extra legs")
    ap.add_argument("--no-graph", action="store_true", help="launch every pass eagerly instead of replaying a CUDA graph")
    ap.add_argument("--unroll", type=int, default=0, help="passes captured per CUDA graph (default: the largest divisor of --steps <= 64)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed pass returned (result records, counts, expansion "
                         "tuples) as DIR/<name>.npy in float32 / float64 (rank 0's shard on several GPUs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


CFG_N = {2: 10_000, 3: 100_000, 4: 100_000, 5: 125_000}
CFG_S = {2: 64, 3: 256, 4: 256, 5: 1024}
CFG_NAME = {2: "configs[1]: 10k StoryRuns x 64 steps, diamond DAG", 3: "configs[2]: 100k StoryRuns x 256 steps, random DAG in-degree 4",
            4: "configs[3]: 100k StoryRuns x 256 steps + condition/gate codes on 50% of steps",
            5: "configs[4]: 1M StoryRuns x 1024 steps with parallel fan-out (8 x 128 branches per run), 125k runs per GPU"}


def algorithmic_bytes(cfg, n_runs, S, E, n_topo, child_nibbles, n_expansion):
    """SURVEY.md 8(d): N*S*(0.75+m) + D*(2(S+1)+2E+S) + N*P*B*0.5 + 8*X."""
    m = 0.5 if cfg in (4,) else 0.0
    state = n_runs * S * (0.75 + m)
    topo = n_topo * (2 * (S + 1) + 2 * E + S)
    child = n_runs * child_nibbles * 0.5
    return state + topo + child + 8 * n_expansion


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.stop_flag, self.ok = [], set(), False, False
        self.active = False
        self.max_mhz = 0
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        nv = self.nv
        mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        if not self.active:
            return
        self.samples.append(mhz)
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                 0x80: "hw_power_brake_slowdown"}
        for bit, n in names.items():
            if r & bit:
                self.reasons.add(n)

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            try:
                self.sample()
            except Exception:
                break
            time.sleep(0.0005)

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz or None, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and so the pinned staging memory it allocates next: first touch, local policy) to the CPUs
    of the NUMA node its GPU hangs off.  Returns a short description or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return "node %d (%d cpus)" % (node, len(allowed))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_inputs(cfg, S, sample_runs):
    """Synthetic sample for the CPU legs, generated without touching bobrapet_b200/lib."""
    from bobrapet_b200 import synth
    from bobrapet_b200.records import layout_py
    from oracle import packed as PK
    gen = os.path.join(ROOT, "oracle", "_build", "libsynth.so")
    if os.path.exists(gen):
        synth.use_library(gen)
    synth.set_threads(min(os.cpu_count() or 1, 32))
    ts = synth.topologies(cfg, 0, sample_runs, S)
    pt = PK.PackedTopologies(ts)
    child = pt.max_child_nibbles()
    fields = (F_COND | F_DECISION if cfg in (4, 5) else 0) | (F_CHILD if child else 0)
    L = layout_py(S, child, fields)
    st = synth.state(cfg, 0, sample_runs, L, np.arange(sample_runs, dtype=np.uint32), ts,
                     pt.child_first[:int(ts.P[0])] if child else None)
    return pt, L, st


def cpu_time(pt, L, st, threads, reps, impl="refshape"):
    """Time a CPU restatement of the reference's per-iteration work on a bounded sample of the workload.

    impl="refshape": oracle/refshape.cc — the reference's own data shapes (string-keyed maps, dependency graph
    rebuilt per pass, buildStateMaps as often as dag.go calls it); impl="packed": oracle/packed_ref.c (bitmask)."""
    from oracle import packed as PK
    times = []
    if impl == "refshape":
        rs = PK.RefShapeBatch(pt, L, st)  # object construction is untimed (the informer cache holds objects)
        rs.run(threads)  # warm
        evals = 0
        for _ in range(reps):
            t0 = time.perf_counter()
            _, evals = rs.run(threads)
            times.append(time.perf_counter() - t0)
        rs.close()
        return evals, times
    PK.evaluate(pt, L, st, 0, 0, threads)  # warm
    for _ in range(reps):
        t0 = time.perf_counter()
        _, counts = PK.evaluate(pt, L, st, 0, 0, threads)
        times.append(time.perf_counter() - t0)
    return counts["evals"], times


def best_thread_count(pt, L, st, cores):
    """"All the host threads it can use": the hash-map-heavy restatement does not scale to every hardware thread on
    every box (allocator contention), so sweep powers of two up to the core count once and keep the fastest."""
    best, best_v, sweep = 1, 0.0, {}
    t = 8
    cands = []
    while t < cores:
        cands.append(t)
        t *= 2
    cands.append(cores)
    for t in cands:
        evals, times = cpu_time(pt, L, st, t, 2, "refshape")
        v = evals / min(times)
        sweep[str(t)] = v
        if v > best_v:
            best, best_v = t, v
    return best, sweep


def reference_arm(args, cfg, S, rank, cores):
    if rank != 0:
        return 0
    sample = args.cpu_sample_runs or min(20_000, 250 * cores)
    pt, L, st = cpu_inputs(cfg, S, sample)
    threads, sweep = best_thread_count(pt, L, st, cores)
    evals, times = cpu_time(pt, L, st, threads, max(args.steps, 1))
    dt = float(np.sum(times))
    v = evals * len(times) / dt
    ev8, t8 = cpu_time(pt, L, st, min(8, cores), 3)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
            "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * dt / len(times), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32 bitmask", "data": "synthetic",
            "config": {"workload": "cfg%d: %d StoryRuns x %d steps per step, a bounded sample of BASELINE configs[%d] (the metric is a rate)" % (cfg, sample, S, cfg - 1),
                       "impl_note": "reference is Go (no toolchain here): reference-shaped C++ restatement oracle/refshape.cc"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "oracle/refshape.cc, %d StoryRuns x %d steps per step, %d threads (fastest of the sweep %s on %d hardware threads)" %
                                       (sample, S, threads, sorted(int(k) for k in sweep), cores),
                             "thread_sweep": sweep,
                             "at_8_threads": ev8 / float(np.median(t8))},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------ GPU arm
class Ctx:
    pass


def graph_unroll(steps, want):
    """Largest divisor of `steps` that is <= want (so the region is whole replays, no eager tail)."""
    want = max(1, min(want, steps))
    for u in range(want, 0, -1):
        if steps % u == 0:
            return u
    return 1


def set_sequence(U, ROT):
    """Input copy used by pass i of a graph: consecutive passes (also across a replay boundary) never share a copy."""
    seq = [i % ROT for i in range(U)]
    if ROT >= 3 and U > 1 and seq[-1] == seq[0]:
        seq[-1] = next(s for s in range(ROT) if s != seq[0] and s != seq[-2])
    return seq


DUMP_BYTES = 60_000_000   # data of all --dump-outputs files together (with the .npy headers: under 64 MB)


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Writes each array of `arrays` (name -> integer array, rows first) as out_dir/<name>.npy: float32 for 8- and 16-bit
    values, float64 for wider ones, so every value is exact.  The smallest arrays go first and each array may use an equal
    share of what the earlier ones left of `budget`; one that does not fit is replaced by a sample of its rows drawn with a
    fixed seed, and the sampled row numbers are written beside it as <name>_rows.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    conv = {k: (np.ascontiguousarray(a), np.float32 if a.dtype.itemsize <= 2 else np.float64) for k, a in arrays.items()}
    left = budget
    for i, name in enumerate(sorted(conv, key=lambda k: conv[k][0].size * np.dtype(conv[k][1]).itemsize)):
        a, ft = conv[name]
        share = left // (len(conv) - i)
        row_bytes = (a.size // max(a.shape[0], 1)) * np.dtype(ft).itemsize
        if a.size * np.dtype(ft).itemsize > share:
            k = share // (row_bytes + 8)
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], size=k, replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
            left -= 8 * k
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(ft))
        left -= a.size * np.dtype(ft).itemsize


def run_config(g, cfg, n_runs, ROT, steps, warmup, reps, headline):
    """Builds the inputs of one configuration on this rank, checks the full batch against the oracle, times it.
    Returns (summary dict, live objects for the headline's extra legs)."""
    import torch
    import torch.distributed as dist
    from bobrapet_b200 import _abi as A, Frontier, synth
    from bobrapet_b200.records import EXP_DTYPE, make_layout
    from bobrapet_b200.sharding import CountExchange, global_offsets
    args, dev, world, rank = g.args, g.dev, g.world, g.rank
    S = CFG_S[cfg]
    # N > 1: one SM is left out of the persistent grid so that the NCCL all-gather of a pass runs beside the next pass
    # instead of queueing behind it (BF_CFG_RESERVE_SMS); BF_BENCH_RESERVE_SMS overrides
    reserve = int(os.environ.get("BF_BENCH_RESERVE_SMS", "1" if world > 1 else "0"))
    fr = Frontier(g.local_rank, reserve_sms=reserve)
    run_lo = rank * n_runs
    fields = A.F_COND | A.F_DECISION if cfg in (4, 5) else 0
    n_topo = args.shared or n_runs
    sets, child, E, parity = [], 0, None, None
    for k in range(ROT):
        ts = synth.topologies(cfg, run_lo + k * 10_000_019, n_topo, S)
        E = int(ts.E[0])
        t_put = time.perf_counter()
        slots = fr.put_topologies(ts)
        if k == 0:
            put_ms = 1e3 * (time.perf_counter() - t_put)
        cf = fr.child_first(int(slots[0])) if int(ts.P[0]) else None
        if cf is not None:
            child = int((int(cf[-1]) + int(ts.parallel["branches"][int(ts.P[0]) - 1]) + 7) // 8 * 8)
        L = make_layout(S, child, fields | (A.F_CHILD if child else 0))
        run_slots = slots if not args.shared else slots[np.arange(n_runs) % n_topo]
        ts_state = ts if not args.shared else synth.topologies(cfg, run_lo + k * 10_000_019, n_runs, S)
        st = synth.state(cfg, run_lo + k * 10_000_019, n_runs, L, run_slots, ts_state, cf)
        d_state = torch.from_numpy(st).to(dev)
        d_result = torch.zeros((n_runs, L.result_stride), dtype=torch.uint8, device=dev)
        d_counts = torch.zeros(4, dtype=torch.int64, device=dev)
        # one untimed pass: its counts size the expansion list (cfg5: the (run, step, branch) tuples of the ready
        # `parallel` steps are emitted in every timed pass, step_executor.go:745-806)
        cur = torch.cuda.current_stream().cuda_stream
        fr.eval_device(L, n_runs, d_state.data_ptr(), d_result.data_ptr(), d_counts.data_ptr(), cur)
        torch.cuda.synchronize()
        got_counts = d_counts.cpu().numpy().tolist()
        exp_cap = int(got_counts[2]) if cfg == 5 else 0
        d_exp = torch.zeros((max(exp_cap, 1), 8), dtype=torch.uint8, device=dev) if exp_cap else None
        sets.append((L, d_state, d_result, d_counts, st if (k == 0 and headline) else None, d_exp, exp_cap))
        if k == 0 and not args.no_parity and not args.shared and not args.ncu:
            # ---- full-size parity (outside every timed region): the whole benchmarked batch of this rank, result
            #      records byte for byte, the counts and the expansion tuples, against oracle/packed_ref.c on the host cores
            from oracle import packed as PK
            if exp_cap:
                d_counts.zero_()
                fr.eval_device(L, n_runs, d_state.data_ptr(), d_result.data_ptr(), d_counts.data_ptr(), cur, flags=A.EVAL_EXPANSION,
                               expansion_ptr=d_exp.data_ptr(), expansion_cap=exp_cap)
                torch.cuda.synchronize()
                got_counts = d_counts.cpu().numpy().tolist()
            got = d_result.cpu().numpy()
            pt = PK.PackedTopologies(ts, slots)
            want, wc = PK.evaluate(pt, L, st, 0, 0, max(1, g.cores // max(world, 1)))
            equal = bool(np.array_equal(got, want)) and got_counts == [wc["ready"], wc["skip"], wc["expansion"], wc["evals"]]
            parity = {"runs": n_runs, "steps": S, "evals": int(wc["evals"]), "records_equal": equal,
                      "oracle": "oracle/packed_ref.c", "oracle_counts": wc}
            if exp_cap:
                wexp, n_wexp = PK.expand(pt, L, st, want, exp_cap)
                gexp = d_exp.cpu().numpy().view(wexp.dtype).reshape(-1)
                parity["expansion_tuples"] = int(n_wexp)
                parity["expansion_equal"] = bool(n_wexp == exp_cap and np.array_equal(gexp, wexp))
                parity["records_equal"] = parity["records_equal"] and parity["expansion_equal"]
                del gexp, wexp
            del got, want, pt
        del ts, ts_state
    L = sets[0][0]
    exch = CountExchange(dev, world)
    gathered = [exch.new_buffer() for _ in range(ROT)]
    work_stream = g.work_stream

    # Consecutive passes work on different batches (ROT disjoint input / result / counts sets), so each pass is submitted with
    # BF_EVAL_COUNTS_SET | BF_EVAL_PIPELINED: no counter fill between passes, and the start-up of pass k + 1 overlaps the tail
    # of pass k (programmatic dependent launch).  BF_BENCH_PIPELINE=0 submits plain passes (fill + kernel, fully serialised).
    pipe_flags = (A.EVAL_COUNTS_SET | A.EVAL_PIPELINED) if (os.environ.get("BF_BENCH_PIPELINE", "1") != "0" and ROT >= 2) else 0

    def one_pass(s, st_, with_gather=True, pf=None):
        pf = pipe_flags if pf is None else pf
        Lk, d_state, d_result, d_counts, _, d_exp, exp_cap = sets[s]
        if not pf:
            d_counts.zero_()
        if exp_cap:
            fr.eval_device(Lk, n_runs, d_state.data_ptr(), d_result.data_ptr(), d_counts.data_ptr(), st_.cuda_stream,
                           flags=A.EVAL_EXPANSION | pf, expansion_ptr=d_exp.data_ptr(), expansion_cap=exp_cap)
        else:
            fr.eval_device(Lk, n_runs, d_state.data_ptr(), d_result.data_ptr(), d_counts.data_ptr(), st_.cuda_stream, flags=pf)
        if world > 1 and with_gather:
            # the path's one collective: all-gather of the per-shard counts, overlapped with the next pass
            exch.gather(d_counts, gathered[s], st_)

    launches0 = fr.stats()["kernel_launches"]
    with torch.cuda.stream(work_stream):
        for i in range(max(warmup, ROT, 3)):
            one_pass(i % ROT, work_stream)
        exch.join(work_stream)
    g.barrier()
    launches_per_pass = (fr.stats()["kernel_launches"] - launches0) / max(warmup, ROT, 3)

    use_graph = not (args.no_graph or args.ncu)
    U = graph_unroll(steps, args.unroll or 64) if use_graph else 1
    seq = set_sequence(U, ROT)

    def capture(with_gather, pf=None):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=work_stream, capture_error_mode="thread_local"):
            for i in range(U):
                one_pass(seq[i], work_stream, with_gather, pf)
            if with_gather:
                exch.join(work_stream)
        with torch.cuda.stream(work_stream):
            gr.replay()  # one untimed replay
        g.barrier()
        return gr

    graph, graph_nc = None, None
    if use_graph:
        try:
            graph = capture(True)
            if world > 1 and headline:
                graph_nc = capture(False)
        except Exception as e:  # capture unsupported: fall back to eager launches
            sys.stderr.write("bench: CUDA graph capture failed (%s); eager launches\n" % e)
            graph, graph_nc, U, seq = None, None, 1, [0]
            g.barrier()

    def region(gr, with_gather):
        if gr is not None:
            for _ in range(steps // U):
                gr.replay()
        else:
            for i in range(steps):
                one_pass(i % ROT, work_stream, with_gather)
            if with_gather:
                exch.join(work_stream)

    def timed(gr, with_gather, n_reps):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_reps)]
        g.barrier()
        g.sampler.active = True
        with torch.cuda.stream(work_stream):
            for a, b in ev:
                g.rendezvous(work_stream)   # device-side: every rank's region starts when the slowest rank arrives
                a.record(work_stream)
                region(gr, with_gather)
                b.record(work_stream)
        g.barrier()
        g.sampler.active = False
        t = torch.tensor([a.elapsed_time(b) for a, b in ev], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().numpy()

    reg = timed(graph, True, reps)
    last = seq[-1] if graph is not None else (steps - 1) % ROT   # the input set of the last timed pass
    outputs = None
    if headline and args.dump_outputs and rank == 0:
        _, _, d_result, d_counts, _, d_exp, exp_cap = sets[last]
        outputs = {"result": d_result.cpu().numpy(), "counts": d_counts.cpu().numpy()}
        if exp_cap:
            e = d_exp.cpu().numpy().view(EXP_DTYPE).reshape(-1)[:min(int(outputs["counts"][2]), exp_cap)]
            outputs["expansion"] = np.stack([e["run"], e["step"], e["branch"]], axis=1).astype(np.uint32)
    ms = float(np.median(reg))
    exposed_us = None
    if graph_nc is not None:
        reg_nc = timed(graph_nc, False, max(3, reps // 2))
        exposed_us = 1e3 * (ms - float(np.median(reg_nc))) / steps
    # the same region with PLAIN passes (counter fill + kernel, every pass waits for the one before): what pipelining buys
    plain_ms = None
    if pipe_flags and graph is not None and fr.stats()["last_kernel"] == 1:   # the pass is the packed-lanes kernel alone: pipelining applies
        try:
            graph_plain = capture(True, 0)
            plain_ms = float(np.median(timed(graph_plain, True, max(3, reps // 2)))) / steps
            del graph_plain
        except Exception as e:
            sys.stderr.write("bench: plain-pass graph failed (%s)\n" % e)
    counts_host = sets[last][3].cpu().numpy().tolist()
    offsets = global_offsets(gathered[last], rank) if world > 1 else None

    # ---- kernel-only duration: event pair around single launches (carries the launch gaps: reported, not used for frac)
    stream = torch.cuda.current_stream()
    kdur = []
    for i in range(min(steps, 30)):
        Lk, d_state, d_result, d_counts = sets[i % ROT][:4]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fr.eval_device(Lk, n_runs, d_state.data_ptr(), d_result.data_ptr(), d_counts.data_ptr(), stream.cuda_stream,
                       flags=A.EVAL_NO_COUNTS)
        b.record(stream)
        torch.cuda.synchronize()
        kdur.append(a.elapsed_time(b))
    kt = torch.tensor([float(np.median(kdur))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(kt, op=dist.ReduceOp.MAX)
    k_ms = float(kt.item())

    abytes = algorithmic_bytes(cfg, n_runs, S, E, n_topo, child, counts_host[2] if cfg == 5 else 0)
    region_ms = ms / steps      # per pass: one frontier_kernel (+ the scan/emit kernels of the expansion when asked for) and
    # one 32-byte counter fill: an upper bound on the kernel's duration.  Pipelined passes OVERLAP (the region per pass is shorter
    # than one launch lasts), so the roofline takes the plain, serialised region: a launch's own duration (+ fill and gap)
    kern_ms = plain_ms if plain_ms else region_ms
    achieved = abytes / (kern_ms * 1e-3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic = tj.get("cfg%d" % cfg, {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    st_stats = fr.stats()
    n_gpus = world if world > 1 else 1
    evals_per_pass = n_runs * S * n_gpus
    out = {
        "workload": "BASELINE %s; %d StoryRuns x %d steps per GPU, %s, E=%d/topology" %
                    (CFG_NAME[cfg], n_runs, S, ("unique topology per run" if not args.shared else "%d shared topologies" % n_topo), E),
        "value": evals_per_pass * steps / (ms * 1e-3), "ms_per_step": ms / steps, "evals_per_pass": evals_per_pass,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": g.peak, "unit": "GB/s", "frac": achieved / g.peak,
                     "traffic": traffic, "traffic_gbs": (traffic / (kern_ms * 1e-3) / 1e9) if traffic else None,
                     "traffic_frac": (traffic / (kern_ms * 1e-3) / 1e9 / g.peak) if traffic else None,
                     "kernel_ms": kern_ms, "kernel_ms_pipelined_region": region_ms if plain_ms else None, "kernel_ms_isolated": k_ms,
                     "frac_at_pipelined_throughput": (abytes / (region_ms * 1e-3) / 1e9 / g.peak) if plain_ms else None,
                     "algorithmic_bytes_per_launch": abytes, "peak_source": g.peak_src,
                     "note": "frac = algorithmic bytes (SURVEY 8(d): canonical u16 CSR + u8 flags + codes) / kernel_ms / peak, kernel_ms = the "
                             "timed region per pass with PLAIN passes (fill + kernel, serialised) — `value` is measured with pipelined passes, "
                             "whose launches overlap (kernel_ms_pipelined_region, frac_at_pipelined_throughput). "
                             "The device adjacency format (fixed-width rows with byte or 10-bit entries, no row_ptr) is SMALLER than the "
                             "canonical figure, so frac can exceed 1: traffic = DRAM bytes ncu measured for one launch of this kernel "
                             "(profiles/ncu_traffic.json), traffic_frac = traffic / the same time / peak = the share of the copy peak the kernel "
                             "really draws. kernel_ms_isolated (event-bracketed single cold launches, max over ranks) is reported beside and not used"},
        "timing": {"region_ms": [float(x) for x in reg], "reps": int(len(reg)), "statistic": "median of the repetitions, each MAX over ranks",
                   "min_ms_per_step": float(np.min(reg)) / steps, "graph_unroll": U if graph is not None else 0,
                   "plain_ms_per_step": plain_ms, "plain_value": (evals_per_pass / (plain_ms * 1e-3)) if plain_ms else None,
                   "plain_note": "the same graph with plain passes (a counter fill + the kernel, fully serialised) instead of pipelined ones",
                   "launches_per_pass": launches_per_pass},
        "collective": None if world == 1 else {"what": "all_gather of 4 x int64 counts per pass, side stream, inside the graph",
                                               "exposed_us": exposed_us, "kernel_ms_max_rank": k_ms},
        "launch": {"grid": st_stats["last_grid"], "block": st_stats["last_block"], "smem": st_stats["last_smem_bytes"],
                   "stages": st_stats["last_stages"], "kernel": st_stats["last_kernel"], "runs_per_trip": st_stats["last_runs_per_trip"],
                   "mode": (("cuda-graph x%d passes, %d replays per region" % (U, steps // U)) if graph is not None else "eager") +
                           ("; passes over the %d rotating batches submitted with BF_EVAL_COUNTS_SET | BF_EVAL_PIPELINED (no fill between "
                            "passes; the start-up of pass k+1 overlaps the tail of pass k where the pass is the packed-lanes kernel alone)" % ROT
                            if pipe_flags else "; plain passes (counter fill + kernel, serialised)"),
                   "pipelined": bool(pipe_flags),
                   "reserved_sms": reserve},
        "parity_check": parity,
        "counts_last_pass": {"ready": counts_host[0], "skip": counts_host[1], "expansion": counts_host[2], "evals": counts_host[3]},
        "global_counts_last_pass": (offsets["total"] if offsets else None),
        "l2": "inputs %.0f MB/pass > 126 MB L2%s" % (abytes / 1e6, (", rotated over %d disjoint copies" % ROT) if ROT > 1 else ""),
    }
    live = Ctx()
    live.fr, live.sets, live.L, live.graph, live.graph_nc = fr, sets, L, graph, graph_nc
    live.timed_launches = int(round(steps * launches_per_pass))
    live.topology_put_ms, live.counts0 = put_ms, counts_host
    live.outputs = outputs
    return out, live


def release(live):
    import gc
    import torch
    live.graph = live.graph_nc = None
    live.sets = None
    gc.collect()
    torch.cuda.synchronize()
    live.fr.close()
    torch.cuda.empty_cache()


def e2e_legs(g, live, n_runs, S, steps):
    """The public host-buffer calls with pinned host memory, copies inside the timed region."""
    import torch
    import torch.distributed as dist
    from bobrapet_b200 import _abi as A
    fr, Lk, dev, world, rank = live.fr, live.L, g.dev, g.world, g.rank
    n_gpus = world if world > 1 else 1
    evals_per_pass = n_runs * S * n_gpus
    state0 = live.sets[0][4]
    hs = fr.alloc_pinned(n_runs * Lk.state_stride).reshape(n_runs, Lk.state_stride)
    hr = fr.alloc_pinned(n_runs * Lk.result_stride).reshape(n_runs, Lk.result_stride)
    hs[:] = state0
    k_e2e = max(5, min(steps, 50))

    def timed_calls(fn):
        for i in range(3):
            fn(i)
        g.barrier()
        t0 = time.perf_counter()
        for i in range(k_e2e):
            fn(i)
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    dt = timed_calls(lambda i: fr.eval(Lk, hs, hr))
    full = {"value": evals_per_pass * k_e2e / dt, "unit": UNIT, "h2d_bytes_per_step": int(n_runs * Lk.state_stride),
            "d2h_bytes_per_step": int(n_runs * Lk.result_stride + 32), "steps": k_e2e,
            "api": "bf_eval (host buffers, synchronous): H2D of every state record + frontier kernel + D2H of every result record"}
    legs = {"full_upload": full}
    # compact results: one head word per run + one 16-bit event per ready / skipped step instead of 80-byte mask records
    ev_cap = int(1.5 * (live.counts0[0] + live.counts0[1])) + 65536
    h_head = fr.alloc_pinned(n_runs * 4).view(np.uint32)
    h_ev = fr.alloc_pinned(ev_cap * 2).view(np.uint16)
    last = [0, 0]

    def call_compact(i):
        r = fr.eval_compact(Lk, hs, ev_cap, head=h_head, events=h_ev)
        last[0] = r[2]
    try:
        dtc = timed_calls(call_compact)
        legs["full_upload_compact"] = {"value": evals_per_pass * k_e2e / dtc, "unit": UNIT, "h2d_bytes_per_step": int(n_runs * Lk.state_stride),
                                       "d2h_bytes_per_step": int(n_runs * 4 + last[0] * 2 + 56), "events_per_step": int(last[0]),
                                       "api": "bf_eval_compact: H2D of every state record + kernels + D2H of one head word per run and 16-bit events"}
    except Exception as ex:
        legs["full_upload_compact"] = {"error": str(ex)[:200]}
    # row f2 — the steady-state tick of the operator: the state stays resident on the device, a tick sends only deltas
    # (1 % of all (run, step) phase codes change per tick: a reconcile is triggered by ONE StepRun changing, 1 / 256 = 0.4 %
    # of a run's codes) and reads the results back
    e2e = None
    try:
        rng = np.random.default_rng(1234 + rank)
        hres = fr.resident_create(Lk, n_runs)
        fr.resident_upload(hres, 0, state0)
        k_delta = max(1, (n_runs * S) // 100)
        dsets = []
        for _ in range(3):
            flat = rng.choice(n_runs * S, size=k_delta, replace=False)
            d = fr.alloc_pinned(k_delta * 8).view(fr.DELTA_DTYPE)       # pinned: the delta upload is asynchronous
            d["run"], d["index"], d["field"] = flat // S, flat % S, A.DELTA_PHASE
            d["code"] = rng.choice([0, 2, 3, 3, 3, 4, 13], size=k_delta)
            dsets.append(d)
        dti = timed_calls(lambda i: fr.resident_tick(hres, Lk, n_runs, dsets[i % 3], hr))
        legs["incremental_dense"] = {"value": evals_per_pass * k_e2e / dti, "unit": UNIT, "change_rate": 0.01,
                                     "h2d_bytes_per_step": int(k_delta * 8), "d2h_bytes_per_step": int(n_runs * Lk.result_stride + 32),
                                     "api": "bf_resident_tick (deltas + pass + mask records, one call): state stays on the device (row f2)"}

        def tick(flags):
            def call(i):
                r = fr.resident_tick_compact(hres, n_runs, dsets[i % 3], ev_cap, flags=flags, head=h_head, events=h_ev)
                last[0], last[1] = r[2], r[4]
            return call
        dtk = timed_calls(tick(0))
        e2e = {"value": evals_per_pass * k_e2e / dtk, "unit": UNIT, "h2d_bytes_per_step": int(k_delta * 8),
               "d2h_bytes_per_step": int(n_runs * 4 + last[0] * 2 + 56), "steps": k_e2e, "change_rate": 0.01,
               "events_per_step": int(last[0]), "runs_listed_per_step": int(last[1]),
               "api": "bf_resident_tick_compact (pinned host buffers, synchronous): the tick's deltas (8 B per changed code) cross PCIe as "
                      "the scatter kernel reads them from the caller's buffer, then the frontier kernel and the on-device compaction, whose "
                      "kernels post one head word per run and one 16-bit event per ready / skipped step of EVERY run straight into the "
                      "caller's buffers (h2d / d2h_bytes_per_step = those bytes; no staging copies on either side)"}
        dtc2 = timed_calls(tick(A.EVAL_CHANGED_ONLY))
        legs["incremental_changed_only"] = {
            "value": evals_per_pass * k_e2e / dtc2, "unit": UNIT, "change_rate": 0.01, "h2d_bytes_per_step": int(k_delta * 8),
            "d2h_bytes_per_step": int(n_runs * 4 + last[0] * 2 + 56), "events_per_step": int(last[0]), "runs_listed_per_step": int(last[1]),
            "api": "bf_resident_tick_compact with BF_EVAL_CHANGED_ONLY: events only for the runs whose result differs from the previous tick's"}
        fr.resident_destroy(hres)
        for d in dsets:
            fr.free_pinned(d.view(np.uint8))
    except Exception as ex:  # never lose the contract line over this leg: fall back to the full-upload figure, flagged
        legs["incremental_error"] = str(ex)[:200]
    if e2e is None:
        e2e = dict(full)
    e2e.update(legs)
    e2e["topology_put_ms"] = live.topology_put_ms
    e2e["topology_put_note"] = ("bf_topology_put_many of this rank's %d topologies (%.0f MB of records), once per Story generation, "
                                "outside the per-tick figure" % (n_runs, live.fr.stats()["arena_used_bytes"] / 3e6))
    fr.free_pinned(h_head.view(np.uint8))
    fr.free_pinned(h_ev.view(np.uint8))
    fr.free_pinned(hs.reshape(-1))
    fr.free_pinned(hr.reshape(-1))
    return e2e


def main():
    args = parse()
    cfg = args.config
    S = CFG_S[cfg]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = world if world > 1 else 1
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        return reference_arm(args, cfg, S, rank, cores)

    # ------------------------------------------------------------------ our arm (GPU)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    import torch
    import torch.distributed as dist
    from bobrapet_b200 import synth

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_MAX_CTAS", "1")   # the collective is 32 bytes per rank: one CTA, so that one reserved SM holds it
        dist.init_process_group("nccl", device_id=dev)
    synth.set_threads(max(1, min(32, len(os.sched_getaffinity(0)) // max(1, min(world, 8)))))
    if args.ncu:
        args.steps, args.warmup, args.no_e2e, args.no_cpu, args.no_extra = min(args.steps, 3), min(args.warmup, 3), True, True, True
    ROT = max(1, args.rot)

    g = Ctx()
    g.args, g.dev, g.world, g.rank, g.local_rank, g.cores = args, dev, world, rank, local_rank, cores
    g.sampler = ClockSampler(local_rank)   # NVML is initialised here, well before any barrier of a timed region
    g.sampler.start()
    g.work_stream = torch.cuda.Stream()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    g.peak = float(peaks.get("hbm_gbs", 6650.0))
    g.peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    token = torch.zeros(1, dtype=torch.int32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def rendezvous(stream):
        if world > 1:
            dist.all_reduce(token)   # enqueued on `stream` (the current stream): later work waits for every rank

    g.barrier, g.rendezvous = barrier, rendezvous

    n_runs = args.runs or CFG_N[cfg]
    head, live = run_config(g, cfg, n_runs, ROT if cfg != 5 else 1, args.steps, args.warmup, max(1, args.reps if not args.ncu else 1), True)
    clocks = g.sampler.result()
    e2e = None
    if not args.no_e2e:
        e2e = e2e_legs(g, live, n_runs, S, args.steps)
    timed_launches, outputs = live.timed_launches, live.outputs
    release(live)

    # ---- the other configurations BASELINE.json names: cfg4 at every N, cfg5 (125k runs x 1024 steps per GPU = 1M x 1024 at 8)
    extra = {}
    if cfg == 3 and not args.no_extra and not args.shared:
        for c2, rot2, steps2 in ((4, ROT, args.steps), (5, 1, max(4, min(args.steps, 20)))):
            try:
                o, lv = run_config(g, c2, CFG_N[c2], rot2, steps2, max(3, args.warmup), max(3, min(args.reps, 7)), False)
                release(lv)
                extra["cfg%d" % c2] = {"workload": o["workload"], "value": o["value"], "ms_per_step": o["ms_per_step"],
                                       "evals_per_pass": o["evals_per_pass"], "frac": o["roofline"]["frac"],
                                       "traffic_frac": o["roofline"]["traffic_frac"], "kernel_ms": o["roofline"]["kernel_ms"],
                                       "plain_ms_per_step": o["timing"]["plain_ms_per_step"],
                                       "achieved_gbs": o["roofline"]["achieved"], "traffic": o["roofline"]["traffic"],
                                       "algorithmic_bytes_per_launch": o["roofline"]["algorithmic_bytes_per_launch"],
                                       "kernel_ms_isolated": o["roofline"]["kernel_ms_isolated"], "steps": steps2,
                                       "region_ms": o["timing"]["region_ms"], "collective": o["collective"], "launch": o["launch"],
                                       "parity_check": o["parity_check"], "counts_last_pass": o["counts_last_pass"],
                                       "global_counts_last_pass": o["global_counts_last_pass"], "l2": o["l2"]}
            except Exception as ex:
                extra["cfg%d" % c2] = {"error": str(ex)[:300]}
    g.sampler.stop_flag = True
    g.sampler.join(timeout=1.0)

    # ---- parity verdict over every rank and every configuration run
    checks = [head["parity_check"]] + [v.get("parity_check") for v in extra.values() if isinstance(v, dict)]
    ok_local = all(c is None or c["records_equal"] for c in checks)
    okt = torch.tensor([1 if ok_local else 0], dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    parity_ok = bool(okt.item())

    # ---- CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if not args.no_cpu and rank == 0 and world == 1:
        sample = args.cpu_sample_runs or min(20_000, 250 * cores)
        pt, Lc, stc = cpu_inputs(cfg, S, sample)
        ev8, t8 = cpu_time(pt, Lc, stc, min(8, cores), 5, "refshape")
        eva, ta = cpu_time(pt, Lc, stc, cores, 5, "refshape")
        evp, tp = cpu_time(pt, Lc, stc, cores, 5, "packed")
        cpu = {"value": ev8 / float(np.median(t8)), "unit": UNIT, "cores": min(8, cores), "kind": "port",
               "sample": "oracle/refshape.cc (reference-shaped: string-keyed maps, per-pass graph rebuild) on %d StoryRuns x %d steps, "
                         "%d threads = the reference's default MaxConcurrentReconciles (controller_config.go:721), median of 5; the Go "
                         "reference itself cannot be built here" % (sample, S, min(8, cores)),
               "all_cores": {"value": eva / float(np.median(ta)), "threads": cores},
               "packed_cpu": {"value": evp / float(np.median(tp)), "threads": cores, "impl": "oracle/packed_ref.c (bitmask)"}}

    rc = 0
    if rank == 0:
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u32 bitmask (integer)", "data": "synthetic",
            "config": {"workload": head["workload"], "l2": head["l2"],
                       "parallelism": "runs sharded across %d GPU(s); one NCCL all-gather of counts per pass" % n_gpus,
                       "grid": head["launch"]["grid"], "block": head["launch"]["block"], "smem": head["launch"]["smem"],
                       "stages": head["launch"]["stages"], "launch": head["launch"]["mode"], "numa": numa},
            "roofline": head["roofline"], "timing": head["timing"], "collective": head["collective"],
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": timed_launches, "clocks": clocks,
            "configs": extra or None,
            "parity_check": dict(head["parity_check"] or {"runs": 0, "records_equal": None}, all_ranks_all_configs_equal=parity_ok),
            "global_counts_last_pass": head["global_counts_last_pass"], "counts_last_pass": head["counts_last_pass"],
        }
        if parity_ok:
            print(json.dumps(line), flush=True)
        else:
            sys.stderr.write("bench: PARITY FAILURE against the oracle; line withheld\n%s\n" % json.dumps(line["parity_check"]))
            rc = 1
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        try:
            dist.barrier(device_ids=[local_rank])
        except Exception:
            pass
        os._exit(rc)
    return rc


if __name__ == "__main__":
    sys.exit(main())
