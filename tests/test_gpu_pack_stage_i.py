"""Stage I of the packed-lanes kernel (frontier_pack.cu) against the packed oracle.  A group whose runs have no compensation or
finally step and none of which takes the realtime + topology-terminated branch computes only the main-group facts; every
other group takes the general code.  The batches here put both kinds of run into one group: main-only runs beside runs with
compensation steps, finally steps, no main step at all, a host group, or realtime + topology-terminated flags; fail-fast runs
with a failed main step, with and without compensation steps; dead and deferred runs.  A group that took the main-only code
while it holds a run that needs the general one gets that run's group, summary or markings wrong.  S = 256 (8 words: 4 runs
per group) and 64 (2 words: 16 runs per group), with and without cond / decision codes.  Exact equality of whole result
records."""
import numpy as np
import pytest

from bobrapet_b200 import _abi as A
from bobrapet_b200 import Frontier
from bobrapet_b200.records import make_layout, pack_state
from oracle import packed as PK
from tests import randgen
from tests.test_gpu_pack_walk import DEAD_SLOT, _merge

pytestmark = pytest.mark.gpu

PHASES = np.array([A.PHASE_NONE, A.PHASE_PENDING, A.PHASE_RUNNING, A.PHASE_SUCCEEDED, A.PHASE_FAILED, A.PHASE_SKIPPED,
                   A.PHASE_PENDING_QUEUED, A.PHASE_TIMEOUT, A.PHASE_COMPENSATED], np.uint8)


@pytest.fixture(scope="module")
def fr():
    f = Frontier(0)
    yield f
    f.close()


def _groups_of(ts):
    off = np.concatenate([[0], np.cumsum(ts.S.astype(np.int64))])
    return [(ts.step_flags[off[i]:off[i + 1]] >> A.SF_GROUP_SHIFT) & 3 for i in range(ts.count)]


def _batch(rng, fr, S, n_groups, fields):
    main_only = randgen.random_topologies(rng, 24, S, S, max_deg=4, groups=False, parallel=False, fill=0.9)
    grouped = randgen.random_topologies(rng, 24, S, S, max_deg=4, groups=True, parallel=False, fill=0.9)
    sf = grouped.step_flags   # the first two grouped topologies: compensation and finally steps only (n_main = 0)
    clear = np.uint8(~np.uint8(3 << A.SF_GROUP_SHIFT) & 0xFF)
    sf[:S // 2] = (sf[:S // 2] & clear) | np.uint8(1 << A.SF_GROUP_SHIFT)
    sf[S // 2:2 * S] = (sf[S // 2:2 * S] & clear) | np.uint8(2 << A.SF_GROUP_SHIFT)
    par = randgen.random_topologies(rng, 4, S, S, max_deg=4, groups=False, parallel=True, fill=0.9)
    ts = _merge(_merge(main_only, grouped), par)
    slots = fr.put_topologies(ts)
    _, child_max = randgen.child_layout(ts)
    L = make_layout(S, child_max, fields | (A.F_CHILD if child_max else 0))
    R = 32 // (1 << (L.words - 1).bit_length())
    n = R * n_groups
    n_plain = main_only.count + grouped.count
    # mostly main-only runs, so that many groups hold main-only runs beside one or two that need the general code
    topo = np.where(rng.random(n) < (0.75 if R == 4 else 0.96), rng.integers(0, main_only.count, size=n), rng.integers(main_only.count, n_plain, size=n))
    deferred = rng.random(n) < 0.03
    topo[deferred] = n_plain + rng.integers(0, par.count, size=int(deferred.sum()))

    phase = PHASES[rng.choice(PHASES.size, size=(n, S), p=[0.3, 0.04, 0.08, 0.4, 0.06, 0.04, 0.04, 0.02, 0.02])]
    done = rng.random(n) < 0.2           # runs whose main steps are all over: the compensation / finally side decides
    phase[done] = np.where(rng.random((int(done.sum()), S)) < 0.8, A.PHASE_SUCCEEDED, A.PHASE_FAILED).astype(np.uint8)
    fail_fast = rng.random(n) < 0.5
    realtime = rng.random(n) < 0.15
    topo_term = rng.random(n) < 0.3
    host = rng.random(n) < 0.05
    rflags = (fail_fast * A.RF_FAIL_FAST | realtime * A.RF_REALTIME | topo_term * A.RF_TOPOLOGY_TERMINATED |
              host * (A.RF_HOST_GROUP | (rng.integers(0, 4, size=n) << A.RF_HOST_GROUP_SHIFT))).astype(np.uint8)
    cond = rng.choice([0, 1, 3], size=(n, S), p=[0.7, 0.15, 0.15]).astype(np.uint8)
    dec = rng.integers(0, 4, size=(n, S)).astype(np.uint8)
    child = np.zeros((n, child_max), np.uint8) if child_max else None
    run_slots = np.asarray(slots)[topo].astype(np.uint32)
    dead = rng.random(n) < 0.02
    run_slots[dead] = DEAD_SLOT
    state = pack_state(L, run_slots, rflags, phase, cond, dec, child)

    # how the groups split: a run needs the general code when its topology has compensation / finally steps or it may take
    # the realtime + topology-terminated branch
    steps_g = _groups_of(ts)
    needs_general = np.array([(steps_g[t] != 0).any() for t in topo]) | (realtime & topo_term)
    needs_general &= ~dead & ~host & ~deferred
    per_group = needs_general.reshape(n_groups, R).sum(axis=1)
    return ts, slots, L, state, dead, per_group, R


@pytest.mark.parametrize("fields", [A.F_ALL_OUT, A.F_COND | A.F_DECISION | A.F_ALL_OUT], ids=["plain", "cond"])
@pytest.mark.parametrize("S", [256, 64])
def test_stage_i_against_oracle(fr, S, fields):
    rng = np.random.default_rng(S * 11 + fields)
    ts, slots, L, state, dead, per_group, R = _batch(rng, fr, S, 1200, fields)
    assert (per_group == 0).sum() > 50 and ((per_group > 0) & (per_group < R)).sum() > 50, np.bincount(per_group)
    got, _ = fr.eval(L, state)   # no validation: dead runs are marked by the kernel
    live_state = state.copy()
    live_state[dead, 0:4] = np.frombuffer(np.uint32(slots[0]).tobytes(), np.uint8)
    want, _ = PK.evaluate(PK.PackedTopologies(ts, slots), L, live_state, threads=8)
    assert (got[dead, 0:4].view("<u4")[:, 0] == 0xFFFFFFFF).all() and not got[dead, 16:].any()
    live = ~dead
    bad = np.nonzero((got[live] != want[live]).any(axis=1))[0]
    assert bad.size == 0, "%d of %d live runs differ from the oracle; first: %d" % (bad.size, int(live.sum()), int(np.nonzero(live)[0][bad[0]]))
    st = fr.stats()
    assert st["last_runs_per_trip"] == R, st   # the packed-lanes kernel took the batch
