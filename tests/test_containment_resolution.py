"""The slow paths of the ordered containment resolution (K1b: k_resolve in containment.cu, k_fabric_resolve in fabric.cu)
against the oracle.

Every victim settles by chasing its open dependencies on an explicit stack.  The chase gives up when the stack is
kChaseDepth deep or after kChaseBudget pushes; the victim then stays open.  Leftovers go round again: whole-grid cooperative
rounds while more than kTailMax are open, then a single block.  Across ranks, victims also wait on foreign piles, in
whole-grid sweeps or, once few are open, one thread per victim.  A bug on any of these paths is silent: k_decode_state
turns whatever state a pile ends in into a death time, so a victim dropped while open dies and its read leaves the graph.

The synth read sets and golden sets never reach these paths: their longest chains of blocking events are about 10 long.
The builder below writes containment structure as RECORDS (chains deeper than the stack, thousands of chains, victims with
hundreds of events, one container of thousands), appended to a small synth read set, so that the whole pipeline runs on
it.  Dovetails tie the designed reads to the background reads, so the edge list and the marks depend on every outcome.

A plain-Python restatement of resolve_victim, run in the order that needs the most rounds, shows on the CPU that the
datasets reach the depth exit, the budget exit and more than kTailMax leftovers, whatever the GPU's scheduling does.
"""
import contextlib
import functools
import time
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import oracle as O
from rala_b200 import api, synth

INF = np.iinfo(np.int64).max

# containment.cu / fabric.cu
K_CHASE_DEPTH, K_CHASE_BUDGET, K_TAIL_MAX = 24, 96, 512
SETTLED, NEVER, DEAD_EVENT = 0x80000000, 0x7FFFFFFF, 0xFFFFFFFF

MARGIN = 15                 # flat piles: [15, L - 15)
CHAIN_LEN = 3000            # length of the bottom read of a chain; every link up is one base longer
DOVE = 1000                 # dovetail overlap length


# ---------------------------------------------------------------------------------------------------------------------
# the builder
# ---------------------------------------------------------------------------------------------------------------------
class Design:
    """Designed reads (lengths, ids from a layout) and designed records in file order, each with the type it must get."""

    def __init__(self, rng):
        self.rng = rng
        self.len = []           # designed read lengths, by designed index
        self.rec = []           # (a, b, a_begin, a_end, b_begin, b_end, flags) with designed indices
        self.want = []          # expected type of each designed record
        self.container = []     # container of each event record (-1: not an event)
        self.chains = []        # designed indices of every chain, bottom (latest event) first

    def read(self, length):
        self.len.append(int(length))
        return len(self.len) - 1

    def contain(self, v, c, kind=None):
        """v contained in c: KB as (v, c, ...) (any lengths), KA as (c, v, ...) (c longer than v)."""
        lv, lc = self.len[v], self.len[c]
        assert lc >= lv
        if kind is None:
            kind = O.KA if lc > lv and self.rng.random() < 0.5 else O.KB
        ori = int(self.rng.integers(0, 2))
        off = MARGIN + int(self.rng.integers(0, lc - lv + 1))    # where v lies inside c's pile
        if kind == O.KB:
            self.rec.append((v, c, MARGIN, lv - MARGIN, off, off + lv - 2 * MARGIN, ori))
        else:
            self.rec.append((c, v, off, off + lv - 2 * MARGIN, MARGIN, lv - MARGIN, ori))
        self.want.append(kind)
        self.container.append(c)

    def self_contain(self, x):
        lx = self.len[x]
        self.rec.append((x, x, MARGIN, lx - MARGIN, MARGIN, lx - MARGIN, 0))
        self.want.append(O.KB)
        self.container.append(x)

    def chain(self, depth, self_every=0):
        """Reverse-time chain x_0 .. x_depth: x_{depth-1} in x_depth first, x_0 in x_1 last.  The outcome alternates down
        the chain (x_{depth-1} dies, x_{depth-2} lives, ...).  Returns the link records in time order, as closures, so
        that several chains can be interleaved."""
        xs = [self.read(CHAIN_LEN + k) for k in range(depth + 1)]
        self.chains.append(xs)
        links = []
        for j in range(depth):
            k = depth - 1 - j
            links.append(functools.partial(self.contain, xs[k], xs[k + 1]))
            if self_every and k % self_every == self_every // 2:   # a self-container right after its own event
                links.append(functools.partial(self.self_contain, xs[k]))
        return xs, links

    def dead_container(self, v, depth):
        """Events that make a fresh container c of v die just before v's event, through a chain of odd depth 1 or 3 below
        it (x_2 in x_3, x_1 in x_2 (x_2 is dead: no effect), c in x_1).  Then the event v in c itself."""
        c = self.read(self.len[v] + 1)
        ups = [c] + [self.read(self.len[v] + 2 + k) for k in range(depth)]
        for k in range(depth - 1, -1, -1):
            self.contain(ups[k], ups[k + 1])
        self.contain(v, c)

    def dovetail(self, x, g, lg):
        """x's suffix overlaps the prefix of background read g: a KAB edge that exists iff both piles survive."""
        lx = self.len[x]
        self.rec.append((x, g, lx - DOVE, lx - MARGIN, MARGIN, DOVE, 0))
        self.want.append(O.KAB)
        self.container.append(-1)
        assert lg > DOVE + MARGIN


def _interleave(rng, seqs):
    """Merge lists of closures keeping each list's order: position-proportional keys with a random tie order."""
    keys, calls = [], []
    for s in seqs:
        n = len(s)
        for i, f in enumerate(s):
            keys.append((i + 0.5) / n + rng.random() * 1e-6)
            calls.append(f)
    for i in np.argsort(keys, kind="stable"):
        calls[i]()


def _family(name, d, rng):
    """Append family `name`'s records to design d."""
    if name == "deep25":
        seqs = [d.chain(25)[1], d.chain(26, self_every=7)[1], d.chain(31)[1]]
        _interleave(rng, seqs)
    elif name == "deep400":
        _interleave(rng, [d.chain(400)[1]])
    elif name == "deep20000":
        _interleave(rng, [d.chain(20_000, self_every=1001)[1], d.chain(60)[1]])
    elif name == "wide":
        # 100 deep: on a B200 the concurrent chases from above settle 40-deep chains within the first sweep
        _interleave(rng, [d.chain(100, self_every=13 if i % 50 == 0 else 0)[1] for i in range(1200)])
    elif name == "wide_fabric":
        _interleave(rng, [d.chain(40, self_every=13 if i % 50 == 0 else 0)[1] for i in range(4800)])
    elif name == "budget":
        for i in range(12):
            v = d.read(CHAIN_LEN - 500)
            for _ in range(int(rng.integers(100, 301))):
                d.dead_container(v, 3 if rng.random() < 0.7 else 1)
            if i % 3 != 2:          # a last event that fires; without it every event found its container dead
                d.contain(v, d.read(CHAIN_LEN))
    elif name == "fanin":
        for hub_depth in (300, 301):          # the hub (bottom of the chain) dies in one, lives in the other
            xs, links = d.chain(hub_depth)
            _interleave(rng, [links])
            hub = xs[0]
            vs = [d.read(CHAIN_LEN - 1 - int(rng.integers(0, 500))) for _ in range(5000)]
            for v in vs:
                d.contain(v, hub)
    else:
        raise KeyError(name)


FAMILIES = ("deep25", "deep400", "deep20000", "wide", "budget", "fanin")
SEEDS = {"deep25": 1, "deep400": 2, "deep20000": 3, "wide": 4, "budget": 5, "fanin": 6, "wide_fabric": 7}


def _layout(n_designed, first, stride):
    """Designed index -> read id.  stride 1: consecutive.  stride S: designed index i goes to block i // S of S ids,
    position i % S... transposed, so that consecutive designed reads (consecutive links of a chain) are S ids apart."""
    if stride == 1:
        return first + np.arange(n_designed)
    rows = (n_designed + stride - 1) // stride       # lanes of `rows` consecutive designed reads each
    i = np.arange(n_designed)
    lane, level = i // rows, i % rows
    return first + level * stride + lane


@functools.lru_cache(maxsize=None)
def build(name, flagged="none", stride=1):
    """Dataset of family `name`: a small synth read set plus the designed reads and records.

    flagged: "none"; "all" (every designed container has a chimeric region, flag 2: the first pass skips their
    containments and the final pass resolves them); "some" (about half of them: first-pass deaths remove final-pass records).
    stride: ids of consecutive designed reads are `stride` apart (32: consecutive links alternate owners under the
    block-cyclic ownership of the multi-GPU session; 32 x world: they stay on one rank)."""
    rng = np.random.Generator(np.random.PCG64(1000 + SEEDS[name]))
    bg = synth.generate(150_000, 6, 5000, seed=SEEDS[name]) if name == "deep400" else \
        synth.generate(300_000, 8, 5000, seed=SEEDS[name])
    n_bg = bg.n_reads
    d = Design(rng)
    first_v, first_c = d.read(CHAIN_LEN), d.read(CHAIN_LEN)      # an event at time 0
    d.contain(first_v, first_c, O.KB)
    _family(name, d, rng)
    last_v, last_c = d.read(CHAIN_LEN), d.read(CHAIN_LEN + 7)    # and one at the last record
    # dovetails from designed reads to background reads, spread over the file
    n_des = len(d.len)
    dv = rng.choice(n_des, size=min(n_des, max(200, n_des // 8)), replace=False)
    tails = [(int(x), int(rng.integers(0, n_bg))) for x in dv]
    des_rec, des_want, des_cont = d.rec, d.want, d.container
    d.rec, d.want, d.container = [], [], []
    for x, g in tails:
        d.dovetail(x, g, int(bg.read_len[g]))
    dov_rec, dov_want, dov_cont = d.rec, d.want, d.container
    d.rec, d.want, d.container = [], [], []
    d.contain(last_v, last_c, O.KA)
    # designed order: the family's records with the dovetails spread over them, then the last event
    pos = np.sort(rng.integers(1, len(des_rec) + 1, len(dov_rec)))
    rec, want, cont = list(des_rec[:1]), list(des_want[:1]), list(des_cont[:1])
    j = 0
    for i in range(1, len(des_rec) + 1):
        while j < len(pos) and pos[j] == i:
            rec.append(dov_rec[j]); want.append(dov_want[j]); cont.append(dov_cont[j])
            j += 1
        if i < len(des_rec):
            rec.append(des_rec[i]); want.append(des_want[i]); cont.append(des_cont[i])
    rec += d.rec; want += d.want; cont += d.container
    n_des = len(d.len)

    # ids: background first, designed reads after it by the layout; one extra unused read if n_piles % 32 == 0
    ids = _layout(n_des, ((n_bg + 31) // 32 * 32) if stride > 1 else n_bg, stride)
    n_piles = int(ids.max()) + 1
    if n_piles % 32 == 0:
        n_piles += 1
    lens = np.full(n_piles, 5000, dtype=np.int64)           # unused ids: reads without records
    lens[:n_bg] = bg.read_len
    lens[ids] = d.len
    # victims at the ends of the id space: swap the first event's victim into id 0 and the last event's victim into id
    # n_piles - 1 (the background reads that held those ids move to theirs)
    perm = np.arange(n_piles)
    for pile, des in ((0, first_v), (n_piles - 1, last_v)):
        other = ids[des]
        perm[[pile, other]] = perm[[other, pile]]
    inv = np.empty_like(perm)
    inv[perm] = np.arange(n_piles)          # old id -> new id
    lens = lens[perm]

    drec = np.array(rec, dtype=np.int64)
    des_b = np.array(want) != O.KAB                      # the dovetails' b ids are background ids already
    drec[:, 0] = ids[drec[:, 0]]
    drec[des_b, 1] = ids[drec[des_b, 1]]
    records = np.empty((bg.n_overlaps + drec.shape[0], 7), dtype=np.int64)
    where = np.sort(rng.choice(np.arange(1, records.shape[0] - 1), size=drec.shape[0] - 2, replace=False))
    is_des = np.zeros(records.shape[0], bool)
    is_des[0] = is_des[-1] = True
    is_des[where] = True
    records[is_des] = drec
    records[~is_des] = bg.records
    records[:, 0], records[:, 1] = inv[records[:, 0]], inv[records[:, 1]]
    records = records.astype(np.uint32)

    piles = np.empty((n_piles, 2), dtype=np.uint32)
    piles[:, 0] = MARGIN
    piles[:, 1] = lens - MARGIN
    flags = np.zeros(n_piles, dtype=np.uint8)
    des_idx = np.nonzero(is_des)[0]
    cont_ids = np.array([inv[ids[c]] if c >= 0 else -1 for c in cont], dtype=np.int64)
    if flagged != "none":
        cs = np.unique(cont_ids[cont_ids >= 0])
        if flagged == "some":
            cs = cs[rng.random(cs.shape[0]) < 0.5]
        flags[cs] = 2
    chains = [inv[ids[np.array(xs)]] for xs in d.chains]
    return SimpleNamespace(name=name, records=records, piles=piles, flags=flags, n_piles=n_piles, n_bg=n_bg,
                           des_idx=des_idx, des_want=np.array(want, dtype=np.uint8), chains=chains,
                           id_first=int(inv[ids[first_v]]), id_last=int(inv[ids[last_v]]))


# ---------------------------------------------------------------------------------------------------------------------
# events, the oracle's death times, the longest blocking chain
# ---------------------------------------------------------------------------------------------------------------------
def first_pass_events(ds):
    """(v, c, t) of the first pass: KA/KB records whose container has no chimeric region, t = file position."""
    rec, types = O.trim_type_batch(ds.records, ds.piles)
    a, b = rec[:, 0].astype(np.int64), rec[:, 1].astype(np.int64)
    kb = (types == O.KB) & ((ds.flags[b] & 2) == 0)
    ka = (types == O.KA) & ((ds.flags[a] & 2) == 0)
    t = np.nonzero(kb | ka)[0]
    return np.where(kb[t], a[t], b[t]), np.where(kb[t], b[t], a[t]), t.astype(np.int64)


def final_pass_events(P):
    """(v, c, t) of the final pass over the oracle's lists after the first pass: t = position in overlaps ++ internals."""
    lst = np.concatenate([P.ovl, P.int])
    _, types = O.trim_type_batch(lst, P.piles)     # the lists hold trimmed records of unchanged piles: trimming is the identity
    a, b = lst[:, 0].astype(np.int64), lst[:, 1].astype(np.int64)
    kb, ka = types == O.KB, types == O.KA
    t = np.nonzero(kb | ka)[0]
    return np.where(kb[t], a[t], b[t]), np.where(kb[t], b[t], a[t]), t.astype(np.int64)


def sequential(v, c, t, n):
    """The reference's loop: an event kills its victim iff victim and container are alive at its time."""
    alive = np.ones(n, bool)
    D = np.full(n, INF)
    for i in np.argsort(t, kind="stable"):
        if alive[v[i]] and alive[c[i]]:
            alive[v[i]] = False
            D[v[i]] = t[i]
    return D


def longest_blocking_chain(v, c, t, n):
    """Longest sequence of events (v, c, t), (c, c', t'), ... with strictly decreasing times: a bound on chase depth."""
    best = np.zeros(n, np.int64)
    o = np.argsort(t, kind="stable")
    vv, cc = v[o], c[o]
    for i in range(vv.shape[0]):
        L = 1 + best[cc[i]]
        if L > best[vv[i]]:
            best[vv[i]] = L
    return int(best.max()) if n else 0


# ---------------------------------------------------------------------------------------------------------------------
# plain-Python restatement of k_resolve
# ---------------------------------------------------------------------------------------------------------------------
class Resolver:
    """resolve_victim and the loops of k_resolve, one victim at a time in a given order."""

    def __init__(self, v, c, t, n):
        o = np.lexsort((t, v))
        self.seg_c = c[o].tolist()
        self.seg_t = t[o].tolist()
        cnt = np.bincount(v, minlength=n)
        self.vstart = np.concatenate([[0], np.cumsum(cnt)]).tolist()
        self.S = [0 if k else SETTLED | NEVER for k in cnt.tolist()]
        self.victims = np.nonzero(cnt)[0]
        self.depth_exits = self.budget_exits = self.dead_events = 0

    def resolve_victim(self, v0):
        S, vstart, seg_c, seg_t = self.S, self.vstart, self.seg_c, self.seg_t
        stack_v, stack_need = [v0], [NEVER]
        budget = K_CHASE_BUDGET
        while stack_v:
            v = stack_v[-1]
            if S[v] & SETTLED:
                stack_v.pop(); stack_need.pop()
                continue
            best_t, best_p = DEAD_EVENT, 0
            for p in range(vstart[v], vstart[v + 1]):
                if seg_t[p] < best_t:
                    best_t, best_p = seg_t[p], p
            if best_t == DEAD_EVENT:                    # every event found its container dead: never killed
                S[v] = max(S[v], SETTLED | NEVER)
                stack_v.pop(); stack_need.pop()
                continue
            S[v] = max(S[v], best_t)
            if best_t > stack_need[-1]:
                stack_v.pop(); stack_need.pop()
                continue
            cn = seg_c[best_p]
            q = SETTLED | NEVER if cn == v else S[cn]
            if q & SETTLED:
                if (q & NEVER) > best_t:
                    S[v] = max(S[v], SETTLED | best_t)
                    stack_v.pop(); stack_need.pop()
                else:
                    seg_t[best_p] = DEAD_EVENT
                    self.dead_events += 1
                continue
            if q > best_t:
                S[v] = max(S[v], SETTLED | best_t)
                stack_v.pop(); stack_need.pop()
                continue
            if len(stack_v) >= K_CHASE_DEPTH:
                self.depth_exits += 1
                return False
            budget -= 1
            if budget <= 0:
                self.budget_exits += 1
                return False
            stack_v.append(cn)
            stack_need.append(best_t)
        return True

    def run(self, order):
        """Cooperative rounds while more than kTailMax are open, then the single-block tail (with its stall detector)."""
        work = list(order)
        rounds, self.left_after_first = 0, None
        while len(work) > K_TAIL_MAX:
            work = [x for x in work if not self.resolve_victim(x)]
            rounds += 1
            if self.left_after_first is None:
                self.left_after_first = len(work)
        stalled, prev = 0, None
        while work:
            stalled = stalled + 1 if prev is not None and len(work) >= prev else 0
            prev = len(work)
            assert stalled <= 64, "the tail stopped shrinking"
            work = [x for x in work if not self.resolve_victim(x)]
            rounds += 1
            if self.left_after_first is None:
                self.left_after_first = len(work)
        self.rounds = rounds
        D = np.array([(s & NEVER) for s in self.S], dtype=np.int64)
        return np.where(D == NEVER, INF, D)


def victim_order(v, t, victims, adversarial=True):
    """Adversarial: victims whose last event is latest first, the bottom of every chain before the links it waits on and
    a victim before the containers of its events.  Otherwise by earliest event: containers before their victims."""
    key = np.full(int(v.max()) + 1, -1 if adversarial else INF)
    (np.maximum if adversarial else np.minimum).at(key, v, t)
    return victims[np.argsort(-key[victims] if adversarial else key[victims], kind="stable")]


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
CASES = [(f, "none") for f in FAMILIES] + [("deep400", "all"), ("wide", "all"), ("wide", "some"), ("budget", "some")]


@functools.lru_cache(maxsize=None)
def oracle_run(name, flagged="none", stride=1):
    ds = build(name, flagged, stride)
    return O.Pipeline(ds.records, ds.piles, ds.flags).run()


@pytest.mark.parametrize("name", FAMILIES + ("wide_fabric",))
def test_designed_records_type_as_intended(name):
    ds = build(name)
    _, types = O.trim_type_batch(ds.records[ds.des_idx], ds.piles)
    bad = np.nonzero(types != ds.des_want)[0]
    assert bad.size == 0, f"{bad.size} designed records type otherwise, first: {ds.records[ds.des_idx[bad[0]]]} " \
                          f"-> {types[bad[0]]}, want {ds.des_want[bad[0]]}"
    assert ds.n_piles % 32 != 0
    v, c, t = first_pass_events(ds)
    assert t[0] == 0 and t[-1] == ds.records.shape[0] - 1, "events at the first and the last record"
    assert ds.id_first == 0 and ds.id_last == ds.n_piles - 1
    assert v[0] == 0 and v[-1] == ds.n_piles - 1, "victims at both ends of the id space"
    if name in ("deep25", "deep20000", "wide", "wide_fabric"):
        assert np.any(v == c), "self-containers inside chains"


def test_layouts_put_links_on_the_owners_they_claim():
    world = 8
    owner = lambda x: (np.asarray(x) // 32) % world           # noqa: E731  (fabric.cuh: pile_owner)
    for stride, alternate in ((32, True), (32 * world, False)):
        ds = build("wide_fabric", "none", stride)
        for xs in ds.chains[:200]:
            o = owner(xs[1:-1])                               # the ends may have been swapped to id 0 / n_piles - 1
            if alternate:
                assert np.all(o[1:] != o[:-1])
            else:
                assert np.all(o == o[0])
        _, types = O.trim_type_batch(ds.records[ds.des_idx], ds.piles)
        assert np.array_equal(types, ds.des_want)


CLAIMED_DEPTH = {"deep25": 25, "deep400": 400, "deep20000": 20_000, "wide": 100, "budget": 4, "fanin": 301}


@pytest.mark.parametrize("name", FAMILIES)
def test_families_reach_the_depths_they_claim(name):
    ds = build(name)
    v, c, t = first_pass_events(ds)
    depth = longest_blocking_chain(v, c, t, ds.n_piles)
    assert depth >= CLAIMED_DEPTH[name], depth
    if name in ("deep25", "deep400", "deep20000", "wide", "fanin"):
        assert depth > K_CHASE_DEPTH
    if name == "deep400":
        assert np.unique(v).size <= K_TAIL_MAX, "every victim fits the single-block tail"
    if name == "wide":
        assert sum(len(xs) - 1 for xs in ds.chains) > 20 * K_TAIL_MAX
    if name == "budget":
        per = np.bincount(v, minlength=ds.n_piles)
        assert np.sum(per >= 100) >= 12 and per.max() <= 301
    if name == "fanin":
        hubs = np.bincount(c, minlength=ds.n_piles)
        assert np.sort(hubs)[-2:].min() >= 5000


def _check_model(v, c, t, n, order_name="adversarial"):
    want = sequential(v, c, t, n)
    R = Resolver(v, c, t, n)
    order = victim_order(v, t, R.victims, order_name == "adversarial")
    got = R.run(order)
    assert np.array_equal(got, want)
    return R, want


@pytest.mark.parametrize("name,flagged", CASES)
def test_model_of_the_resolver_reaches_the_oracle(name, flagged):
    """The restated resolver ends in the sequential death times, and in the oracle's piles, on the first pass and on the
    final pass.  A 20 000-deep chain in the adversarial order needs ~830 sweeps of the whole chain (quadratic work in
    Python), so that dataset runs its worklist containers first; the tail and the cooperative rounds are shown on the others."""
    ds = build(name, flagged)
    P = oracle_run(name, flagged)
    v, c, t = first_pass_events(ds)
    R, D = _check_model(v, c, t, ds.n_piles, "containers first" if name == "deep20000" else "adversarial")
    after_first = O.Pipeline(ds.records, ds.piles, ds.flags).classify()
    assert np.array_equal(D != INF, after_first.piles[:, 1] == 0)
    if flagged != "none":
        fv, fc, ft = final_pass_events(after_first.retrim())
        assert ft.shape[0] > 100
        Rf, Df = _check_model(fv, fc, ft, ds.n_piles)
        assert np.array_equal((D != INF) | (Df != INF), P.piles[:, 1] == 0)
        R = SimpleNamespace(**{k: getattr(Rf, k) + (getattr(R, k) if flagged == "some" else 0)   # counters of both passes
                               for k in ("depth_exits", "budget_exits", "dead_events", "rounds")},
                            left_after_first=Rf.left_after_first)
        v, D = (np.concatenate([v, fv]), np.minimum(D, Df)) if flagged == "some" else (fv, Df)
    else:
        assert np.array_equal(D != INF, P.piles[:, 1] == 0)
    if flagged == "some":           # first-pass deaths took records of flagged containers out of the final pass
        rec, types = O.trim_type_batch(ds.records, ds.piles)
        cont = np.where(types == O.KB, rec[:, 1], rec[:, 0])
        skipped = np.isin(types, (O.KA, O.KB)) & ((ds.flags[cont] & 2) != 0)
        assert skipped.sum() > ft.shape[0] + 100
        return
    if name in ("deep25", "deep400", "wide", "fanin"):
        assert R.depth_exits > 0
    if name == "budget":
        assert R.budget_exits > 0 and R.dead_events > 0
        never = np.nonzero((np.bincount(v, minlength=ds.n_piles) >= 100) & (D == INF))[0]
        assert never.size >= 1, "a victim whose events all find dead containers"
    if name == "wide" and flagged != "some":
        assert R.left_after_first > K_TAIL_MAX
    if name == "deep400":
        assert R.rounds >= 2


def test_model_paths_on_the_reverse_chain():
    """x_{n-1} in x_n at time 0, ..., x_0 in x_1 at time n - 1: alive, dead, alive, ... from x_0; every exit is taken."""
    n = 50
    x = np.arange(n + 1)
    v = x[:-1][::-1].copy()
    c = v + 1
    t = np.arange(n)
    R, D = _check_model(v, c, t, n + 1)
    assert [bool(D[k] != INF) for k in range(n)] == [(n - 1 - k) % 2 == 0 for k in range(n)]
    assert R.depth_exits > 0 and R.rounds >= 2


# ---------------------------------------------------------------------------------------------------------------------
# GPU: one device
# ---------------------------------------------------------------------------------------------------------------------
def _same_graph(G, P, label):
    c = G.counts()
    assert np.array_equal(G.piles(), P.piles), f"{label}: piles"
    ovl, inl = G.lists()
    assert np.array_equal(ovl, P.ovl), f"{label}: final overlaps"
    assert np.array_equal(inl, P.int), f"{label}: final internals"
    assert np.array_equal(G.edges(), P.edges), f"{label}: edges"
    assert np.array_equal(G.marked(), P.marked), f"{label}: marks"
    assert np.array_equal(G.seq_to_node(), P.seq_to_node), f"{label}: node ids"
    assert c["n_nodes"] == P.n_nodes and c["n_edges"] == P.edges.shape[0] and c["n_transitive_pairs"] == P.n_pairs, label
    return c


NEED_ROUNDS = {"deep400", "deep20000", "wide"}


@contextlib.contextmanager
def _closing(session):
    """A session is closed whatever the test finds: several ranks' arenas must not outlive a failed comparison."""
    try:
        yield session
    finally:
        session.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,flagged", CASES)
def test_resolution_eager_captured_replayed(ctx, name, flagged):
    ds = build(name, flagged)
    P = oracle_run(name, flagged)
    with _closing(api.Graph(ctx)) as G:
        G.use_cuda_graph(False)
        G.set_piles(ds.piles, ds.flags).set_hills(None).set_overlaps(ds.records)
        G.run()
        seen = [_same_graph(G, P, "eager")]
        G.use_cuda_graph(True)
        for i in range(3):   # eager (shape seen), captured + launched, replayed
            G.run()
            seen.append(_same_graph(G, P, f"graph run {i}"))
    rounds = [s["n_rounds"] for s in seen]
    final_rounds = [s["n_final_rounds"] for s in seen]
    print(f"\n{name}/{flagged}: n_rounds {rounds}, n_final_rounds {final_rounds}")
    if name in NEED_ROUNDS and flagged == "none":
        assert min(rounds) >= 2, rounds
    if flagged == "all" and name in NEED_ROUNDS:
        assert min(final_rounds) >= 2, final_rounds


# ---------------------------------------------------------------------------------------------------------------------
# GPU: several ranks of the multi-GPU session on one device
# ---------------------------------------------------------------------------------------------------------------------
def _check_multi(M, P, label):
    c = M.counts()
    edges, marked = M.all_edges()
    assert np.array_equal(edges, P.edges), f"{label}: edge list"
    assert np.array_equal(marked, P.marked), f"{label}: removed-edge set"
    assert np.array_equal(M.piles(), P.piles), f"{label}: pile liveness"
    assert np.array_equal(M.seq_to_node(), P.seq_to_node), f"{label}: node ids"
    assert c["n_transitive_pairs"] == P.n_pairs and c["n_nodes"] == P.n_nodes and c["n_edges"] == P.edges.shape[0], label
    return c


def _stride(layout, world):
    return 32 if layout == "alternating" else 32 * world


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("layout", ["alternating", "rank_local"])
def test_fabric_resolution_matches_the_oracle(world, layout):
    stride = _stride(layout, world)
    ds = build("wide", "none", stride)
    P = oracle_run("wide", "none", stride)
    with _closing(api.Multi([0] * world)) as M:
        M.set_piles(ds.piles, ds.flags).set_shards(ds.records).plan()
        M.use_cuda_graph(False)
        M.run()
        seen = [_check_multi(M, P, f"world {world} {layout} eager")]
        M.use_cuda_graph(True)
        for i in range(3):
            M.run()
            seen.append(_check_multi(M, P, f"world {world} {layout} graph run {i}"))
        sweeps = [len(M.sweep_log(k, 0)) for k in range(world)]
    print(f"\nworld {world} {layout}: n_rounds {[s['n_rounds'] for s in seen]}, "
          f"n_final_rounds {[s['n_final_rounds'] for s in seen]}, first-pass sweeps per rank {sweeps}")
    assert min(s["n_rounds"] for s in seen) >= 2


FABRIC_FAMILIES = [("deep20000", "none", "alternating"), ("fanin", "none", "alternating"), ("budget", "none", "rank_local"),
                   ("deep400", "all", "alternating"), ("wide", "some", "alternating"), ("budget", "some", "rank_local")]


@pytest.mark.gpu
@pytest.mark.parametrize("name,flagged,layout", FABRIC_FAMILIES)
def test_fabric_families_match_the_oracle(name, flagged, layout):
    """The other families across three ranks: a 20 000-link chain whose links alternate owners, thousands of victims of
    one container, victims that run out of chase budget on their own rank, and final passes that resolve chains."""
    world = 3
    stride = _stride(layout, world)
    ds = build(name, flagged, stride)
    P = oracle_run(name, flagged, stride)
    with _closing(api.Multi([0] * world)) as M:
        M.set_piles(ds.piles, ds.flags).set_shards(ds.records).plan()
        M.use_cuda_graph(False)
        M.run()
        seen = [_check_multi(M, P, f"{name}/{flagged} eager")]
        M.use_cuda_graph(True)
        for i in range(2):   # captured + launched, replayed
            M.run()
            seen.append(_check_multi(M, P, f"{name}/{flagged} graph run {i}"))
        sweeps = [[len(M.sweep_log(k, p)) for k in range(world)] for p in (0, 1)]
    print(f"\n{name}/{flagged} world 3 {layout}: n_rounds {[s['n_rounds'] for s in seen]}, "
          f"n_final_rounds {[s['n_final_rounds'] for s in seen]}, sweeps per rank (first, final pass) {sweeps}")
    if flagged == "none":
        assert seen[0]["n_candidates"] > 0
    if flagged == "all":
        assert min(s["n_final_rounds"] for s in seen) >= 2


@pytest.mark.gpu
def test_fabric_whole_grid_sweeps_and_too_few_rounds():
    """At world 8 the resolution grid of a rank is 1/16 of the device: the wide family leaves more victims open than it
    has threads, so it runs whole-grid sweeps before the poll phase.  With one sweep allowed, some ranks give up while
    others already watch single victims: the step must end on every rank, say that it did not fit (or be right), and a
    new plan() must recover the oracle's answer."""
    world = 8
    ds = build("wide_fabric", "none", 32)
    P = oracle_run("wide_fabric", "none", 32)
    with _closing(api.Multi([0] * world)) as M:
        M.set_piles(ds.piles, ds.flags).set_shards(ds.records).plan()
        M.run()
        c = _check_multi(M, P, "plan")
        logs = [M.sweep_log(k, 0) for k in range(world)]
        print(f"\nwide_fabric world 8: n_rounds {c['n_rounds']}, sweeps per rank {[len(lg) for lg in logs]}, "
              f"open victims per sweep on rank 0 {logs[0][:, 0].tolist()}")
        # every sweep log entry but the poll phase's is a whole-grid sweep; at least two of them on some rank
        assert max(len(lg) for lg in logs) >= 3, [len(lg) for lg in logs]
        assert c["n_rounds"] >= 3
        M.set_rounds(1, 1)
        t0 = time.perf_counter()
        M.run().synchronize()
        seconds = time.perf_counter() - t0
        need, fits = M.demand()
        logs = [M.sweep_log(k, 0) for k in range(world)]
        print(f"one sweep allowed: fits {fits}, {seconds:.3f} s, rounds asked for {int(need[3])}, "
              f"sweeps per rank {[len(lg) for lg in logs]}")
        assert seconds < 2.0, "a rank waited for a peer that had given up"
        if fits:
            _check_multi(M, P, "one round, reported as fitting")
        else:
            with pytest.raises(api.RalaB200Error):
                M.counts()
        M.plan()
        M.run()
        _check_multi(M, P, "re-planned")
