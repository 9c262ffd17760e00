"""The packed-lanes kernel's dependency walk and status bytes (frontier_pack.cu) against the packed oracle, on batches
built around them: groups of four runs with 0, 1, 2, 3, 5 and 32 walked (run, word) items (the 4 / 2 / 1 remainders of the
walk), runs with and without a failed-dependency class side by side in one group, pending steps without needs, dead and
deferred runs inside a group, and cond FAIL codes (the fix-up loop after the walk).  S = 129 ... 256 takes the 8-word
byte-row path; 64 and 300 the other fixed-width paths.  Exact equality of whole result records."""
import numpy as np
import pytest

from bobrapet_b200 import _abi as A
from bobrapet_b200 import Frontier
from bobrapet_b200.frontier import TopologySet
from bobrapet_b200.records import make_layout, pack_state
from oracle import packed as PK
from tests import randgen

pytestmark = pytest.mark.gpu

ITEMS = (0, 1, 2, 3, 5, 32)   # walked (run, word) items per group, cycled over the groups of a batch
DEAD_SLOT = 0x7FFFFFF0


@pytest.fixture(scope="module")
def fr():
    f = Frontier(0)
    yield f
    f.close()


def _merge(a: TopologySet, b: TopologySet) -> TopologySet:
    """a's topologies, then b's (b's parallel descriptors point past a's branch-allow bits)"""
    bits_a = np.unpackbits(a.allow_bits, bitorder="little") if a.allow_bits.size else np.zeros(0, np.uint8)
    bits_b = np.unpackbits(b.allow_bits, bitorder="little") if b.allow_bits.size else np.zeros(0, np.uint8)
    par_b = b.parallel.copy()
    par_b["allow_first"] += bits_a.size
    bits = np.concatenate([bits_a, bits_b])
    allow = np.packbits(bits, bitorder="little") if bits.size else None
    par = np.concatenate([a.parallel, par_b])
    return TopologySet(np.concatenate([a.S, b.S]), np.concatenate([a.E, b.E]), np.concatenate([a.row_ptr, b.row_ptr]),
                       np.concatenate([a.col_idx, b.col_idx]), np.concatenate([a.step_flags, b.step_flags]),
                       np.concatenate([a.P, b.P]), par if par.size else None, allow)


def _batch(rng, fr, S, n_groups, fields):
    plain = randgen.random_topologies(rng, 40, S, S, max_deg=4, groups=False, parallel=False, fill=0.9)
    par = randgen.random_topologies(rng, 4, S, S, max_deg=4, groups=False, parallel=True, fill=0.9)
    ts = _merge(plain, par)
    slots = fr.put_topologies(ts)
    _, child_max = randgen.child_layout(ts)
    L = make_layout(S, child_max, fields | (A.F_CHILD if child_max else 0))
    W = (S + 31) // 32
    n = 4 * n_groups
    topo = rng.integers(0, plain.count, size=n)
    deferred = rng.random(n) < 0.03
    topo[deferred] = plain.count + rng.integers(0, par.count, size=int(deferred.sum()))
    rp = np.split(ts.row_ptr, np.cumsum(ts.S.astype(np.int64) + 1)[:-1])
    has_needs = [np.diff(r.astype(np.int64)) > 0 for r in rp]

    fail_fast = rng.random(n) < 0.5
    phase = np.full((n, S), A.PHASE_SUCCEEDED, np.uint8)
    # failed steps only in runs without fail-fast: there they give the run a failed-dependency class and keep its candidates
    failed = (rng.random((n, S)) < 0.04) & ~fail_fast[:, None]
    phase[failed] = A.PHASE_FAILED
    for q in range(n_groups):
        pairs = rng.choice(4 * W, size=min(ITEMS[q % len(ITEMS)], 4 * W), replace=False)
        for pr in pairs:
            r, w = 4 * q + int(pr) // W, int(pr) % W
            steps = np.arange(w * 32, min(S, w * 32 + 32))
            steps = steps[has_needs[topo[r]][steps]]
            if steps.size:   # a word without a step that has needs cannot be walked
                pick = rng.choice(steps, size=min(steps.size, int(rng.integers(1, 5))), replace=False)
                phase[r, pick] = A.PHASE_NONE
        # candidates without needs: met without a walk
        r = 4 * q + int(rng.integers(0, 4))
        free = np.nonzero(~has_needs[topo[r]])[0]
        phase[r, free[:2]] = A.PHASE_NONE
    cond = rng.choice([0, 1, 3], size=(n, S), p=[0.7, 0.15, 0.15]).astype(np.uint8)
    dec = rng.integers(0, 4, size=(n, S)).astype(np.uint8)
    rflags = fail_fast.astype(np.uint8) * A.RF_FAIL_FAST
    child = np.zeros((n, child_max), np.uint8) if child_max else None
    run_slots = np.asarray(slots)[topo].astype(np.uint32)
    dead = rng.random(n) < 0.02
    run_slots[dead] = DEAD_SLOT
    state = pack_state(L, run_slots, rflags, phase, cond, dec, child)
    return ts, slots, L, state, dead


@pytest.mark.parametrize("fields", [A.F_ALL_OUT, A.F_COND | A.F_DECISION | A.F_ALL_OUT], ids=["plain", "cond"])
@pytest.mark.parametrize("S", [129, 200, 255, 256, 64, 300])
def test_walk_against_oracle(fr, S, fields):
    rng = np.random.default_rng(S * 7 + fields)
    ts, slots, L, state, dead = _batch(rng, fr, S, 1500, fields)
    got, _ = fr.eval(L, state)   # no validation: dead runs are marked by the kernel
    live_state = state.copy()
    live_state[dead, 0:4] = np.frombuffer(np.uint32(slots[0]).tobytes(), np.uint8)
    want, _ = PK.evaluate(PK.PackedTopologies(ts, slots), L, live_state, threads=8)
    assert (got[dead, 0:4].view("<u4")[:, 0] == 0xFFFFFFFF).all() and not got[dead, 16:].any()
    live = ~dead
    bad = np.nonzero((got[live] != want[live]).any(axis=1))[0]
    assert bad.size == 0, "%d of %d live runs differ from the oracle; first: %d" % (bad.size, int(live.sum()), int(np.nonzero(live)[0][bad[0]]))
    st = fr.stats()
    assert st["last_runs_per_trip"] == 32 // (1 << (L.words - 1).bit_length()), st   # the packed-lanes kernel took the batch
