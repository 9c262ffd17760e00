"""Device groups through the C ABI (bf_group_*): one process, G GPUs, runs sharded in contiguous blocks, one NCCL
all-gather of the per-shard counts per pass, and limiters whose totals are all-reduced across the shards.

On a 1-GPU box the group has one shard (the communicator has one rank); with 2+ GPUs every G up to the device count runs."""
import functools

import numpy as np
import pytest
import torch  # before any group exists: bf_group_create dlopens libnccl.so.2, and torch must load its own build of it first

from bobrapet_b200 import _abi as A
from bobrapet_b200 import FrontierGroup, synth
from bobrapet_b200.records import make_layout
from oracle import limiters as LM
from oracle import packed as PK
from tests import randgen
from tests.test_gpu_limiters import _running_and_demand

pytestmark = pytest.mark.gpu


# Group sizes are fixed here rather than read from the box, so that a test has the same ids on every machine: the one-device
# variants run wherever there is a GPU, and test_groups_of_several_devices runs the same checks on 2, 3, 4 and 8 devices.
@pytest.fixture(params=[1])
def group(request):
    g = FrontierGroup(list(range(request.param)))
    yield g
    g.close()


def test_group_eval_sharded_topologies(group):
    """unique-topology mode: every shard holds the topologies of its own block of runs (slot ids are per shard)"""
    n, S = 9001, 256
    ts_all = synth.topologies(4, 0, n, S)
    L = make_layout(S, 0, A.F_COND | A.F_DECISION | A.F_ALL_OUT)
    state = np.zeros((n, L.state_stride), dtype=np.uint8)
    want = np.zeros((n, L.result_stride), dtype=np.uint8)
    per_want = []
    covered = 0
    for k in range(group.size):
        first, count = group.shard_range(n, k)
        assert first == covered
        covered += count
        if count == 0:
            per_want.append({"ready": 0, "skip": 0, "expansion": 0, "evals": 0})
            continue
        ts = synth.topologies(4, first, count, S)
        slots = group.shards[k].put_topologies(ts)
        state[first:first + count] = synth.state(4, first, count, L, slots, ts)
        want[first:first + count], wc = PK.evaluate(PK.PackedTopologies(ts, slots), L, state[first:first + count], threads=8)
        per_want.append(wc)
    assert covered == n
    got, counts, per = group.eval(L, state)
    assert np.array_equal(got, want)
    assert per == per_want
    assert counts == {f: sum(p[f] for p in per_want) for f in ("ready", "skip", "expansion", "evals")}


@pytest.mark.parametrize("seed", range(3))
def test_group_schedule_holds_limits_across_shards(group, seed):
    """replicated topologies; limits, bases and priority ordering are enforced over the WHOLE batch, not per shard"""
    rng = np.random.default_rng(8100 + seed)
    ts = randgen.random_topologies(rng, 30, 1, [60, 257, 130][seed], parallel=(seed == 0))
    slots = group.put_topologies_replicated(ts)
    n = [3001, 2500, 4003][seed]
    L, state, topo = randgen.random_state(rng, ts, slots, n, A.F_COND | A.F_DECISION, phase_mix=("any" if seed % 2 else "progress"))
    want, wcounts = PK.evaluate(PK.PackedTopologies(ts, slots), L, state, threads=8)
    result, counts, _ = group.eval(L, state)
    assert np.array_equal(result, want) and counts == wcounts
    W = L.words
    ready = np.ascontiguousarray(result[:, L.off_ready:L.off_ready + 4 * W]).view("<u4").reshape(n, W)
    n_stories, n_queues = int(rng.integers(1, 20)), int(rng.integers(1, 5))
    sched = np.zeros(n, dtype=LM.SCHED_RUN_DTYPE)
    sched["story_key"] = rng.integers(0, n_stories, size=n)
    sched["queue_key"] = rng.integers(0, n_queues, size=n)
    sched["priority"] = rng.integers(-3, 8, size=n)
    el = rng.integers(0, 4000, size=n).astype(np.uint32)
    el[rng.random(n) < 0.5] = LM.NONE_U32
    sched["queued_elapsed_s"] = el
    sched["run_phase"] = rng.choice([0, 1, 2, 3, 4, 8, 11], size=n)
    story_limit = rng.choice([0, 0, 1, 3, 40, 200, 1000], size=n_stories).astype(np.int32)
    queue_limit = rng.choice([0, 50, 2000, 20000], size=n_queues).astype(np.int32)
    queue_aging = rng.choice([0, 30, 60, 600], size=n_queues).astype(np.int32)
    global_limit = int(rng.choice([0, 100, 5000, 100000]))
    story_base = rng.integers(0, 5, size=n_stories).astype(np.uint32)
    queue_base = rng.integers(0, 50, size=n_queues).astype(np.uint32)
    global_base = int(queue_base.sum())
    got = group.schedule(L, n, sched, story_limit, queue_limit, queue_aging, global_limit, story_base, queue_base, global_base)
    run_running, run_demand = _running_and_demand(ts, topo, L, state)
    launch, q_story, q_sched, info, sr, qr, gr, mp = LM.schedule_packed(
        run_running, run_demand, sched, ready, story_limit, story_base, queue_limit, queue_aging, queue_base, global_limit, global_base)
    assert np.array_equal(got["story_running"], sr.astype(np.uint32)) and np.array_equal(got["queue_running"], qr.astype(np.uint32))
    assert got["global_running"] == gr and np.array_equal(got["queue_max_priority"].astype(np.int64), mp)
    rec = got["records"]
    masks = np.ascontiguousarray(rec[:, 16:16 + 12 * W]).view("<u4").reshape(n, 3, W)
    assert np.array_equal(masks[:, 0], launch) and np.array_equal(masks[:, 1], q_story) and np.array_equal(masks[:, 2], q_sched)
    assert np.array_equal(np.ascontiguousarray(rec[:, 0:16]).view("<u4").reshape(n, 4), info)


def test_group_rejects_bad_arguments(group):
    L = make_layout(32, 0, 0)
    with pytest.raises(A.FrontierError):
        group.schedule(L, 5, np.zeros(5, dtype=LM.SCHED_RUN_DTYPE), [0], [0], [0])   # no preceding bf_group_eval of 5 runs
    import ctypes as C
    lib = A.load()
    g = C.c_void_p()
    dup = (C.c_int32 * 2)(0, 0)
    assert lib.bf_group_create(C.byref(g), dup, 2, None) == A.BF_EINVAL          # the same device twice
    assert lib.bf_group_create(C.byref(g), dup, 0, None) == A.BF_EINVAL


def test_groups_of_several_devices():
    """the group tests above on every group of 2, 3, 4 and 8 devices the box holds, a fresh group for each check"""
    sizes = [n for n in (2, 3, 4, 8) if n <= torch.cuda.device_count()]
    if not sizes:
        pytest.skip("needs at least 2 GPUs")
    checks = [test_group_eval_sharded_topologies, test_group_rejects_bad_arguments] + \
             [functools.partial(test_group_schedule_holds_limits_across_shards, seed=s) for s in range(3)]
    for n in sizes:
        for check in checks:
            g = FrontierGroup(list(range(n)))
            try:
                check(g)
            finally:
                g.close()


def test_queue_max_priority_base_blocks_lower_priority_runs():
    """bf_sched_tables.queue_max_priority_base: a higher-priority run with demand OUTSIDE the batch queues the batch's
    lower-priority runs (enforcePriorityOrdering compares against every non-terminal StoryRun of the queue, dag.go:1917-1944;
    dag_test.go:528 TestEnforcePriorityOrderingBlocksLowerPriority)"""
    from bobrapet_b200 import Frontier
    f = Frontier(0)
    try:
        ts = synth.topologies(3, 0, 16, 64)
        slots = f.put_topologies(ts)
        L = make_layout(64, 0, 0)
        state = np.zeros((16, L.state_stride), dtype=np.uint8)
        state[:, 0:4] = np.ascontiguousarray(slots, dtype="<u4").view(np.uint8).reshape(16, 4)
        result, counts = f.eval(L, state)               # nothing started: the steps without needs are ready
        assert counts["ready"] >= 16
        sched = np.zeros(16, dtype=LM.SCHED_RUN_DTYPE)
        sched["priority"], sched["queued_elapsed_s"], sched["run_phase"] = 1, LM.NONE_U32, 2
        free = f.schedule(L, 16, sched, [0], [0], [0])
        blocked = f.schedule(L, 16, sched, [0], [0], [0], queue_max_priority_base=[5])
        equal = f.schedule(L, 16, sched, [0], [0], [0], queue_max_priority_base=[1])
        hdr = lambda r: np.ascontiguousarray(r["records"][:, 0:16]).view("<u4").reshape(16, 4)
        assert (hdr(free)[:, 0] > 0).all() and (hdr(free)[:, 2] == 0).all()
        assert (hdr(blocked)[:, 0] == 0).all() and (hdr(blocked)[:, 3] == A.QUEUED_PRIORITY).all() and int(blocked["queue_max_priority"][0]) == 5
        assert np.array_equal(hdr(equal), hdr(free))    # an equal priority outside does not outrank (strictly greater, :1933)
    finally:
        f.close()
