"""Parity of the CUDA path with the CPU oracle across the launch geometries, node-count regimes, kernel variants and
resource-vector widths the host chooses between (vcalloc.cu choose_geometry, the commit / backfill / dense / evict
launchers). Every other GPU file runs a handful of fixed cluster shapes; here each case names the branch it exists for
and asserts, through expected_geometry, that it still lands there. Results are compared bit for bit, fp64 scores
included. The file sorts after every other GPU file on purpose: the suite runs with -x, and a kernel fault poisons
the CUDA context, so a failure here cannot hide the results of the older files."""
import contextlib
import dataclasses
import importlib.util
import os
import random

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

VC_KERNEL_GENERAL, VC_KERNEL_INCREMENTAL = 0, 1


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def expected_geometry(N, sm, fast, ctas=0, threads=0):
    """(G, npc, block) of the commit kernels for N nodes on one GPU with `sm` SMs: a plain restatement of
    choose_geometry (volcano_b200/csrc/vcalloc.cu). `fast`: the incremental kernel (k_commit_fast) serves the session;
    `ctas` / `threads`: VC_COMMIT_CTAS / VC_COMMIT_THREADS (0 = unset)."""
    g = ctas if ctas > 0 else sm
    block = max(128, min(256, threads // 32 * 32)) if threads > 0 else 128
    g = max(1, min(g, (N + 31) // 32))  # at least a warp of nodes per CTA
    npc = max(32, (-(-N // g) + 31) // 32 * 32)
    if fast and ctas <= 0 and npc < 128 and N >= 64 * 128:  # mid-sized clusters: four full warps of nodes per CTA
        npc = 128
    G = max(1, -(-N // npc))
    if npc > block:
        block = min(256, (npc + 31) // 32 * 32)
    if fast and threads <= 0:
        block = 256
    return G, npc, block


# sizeof(Ctl) / sizeof(CtlFast) of vc_commit.cuh / vc_commit_fast.cuh (host compile for sm_100a)
CTL_BYTES, CTLFAST_BYTES = 3864, 3488


def commit_smem(npc, G, R, K, fast, future, nta_L=0):
    """Dynamic shared memory of one commit CTA without the queue heaps: a restatement of the estimate at the end of
    choose_geometry. `future`: Releasing / Pipelined rows, a topology job or feasible-node sampling (dc.has_future).
    The incremental kernel adds the heaps only while the total stays under 200 KB, so this decides whether a
    geometry fits the device at all."""
    a16 = lambda x: (x + 15) & ~15  # noqa: E731
    if fast:
        rows = 3 * R + (2 * R if future else 0) + 2 * K + 2 + 1
        return a16(CTL_BYTES) + a16(CTLFAST_BYTES) + rows * npc * 8 + npc * (8 + 4 * 5) + G * (8 + 4 + 4 + 4 + 4) + 64
    rows = 3 * R + (2 * R if future else 0) + 2 * K + 2
    b = a16(CTL_BYTES) + rows * npc * 8 + npc * (8 + 4 + 4) + 64 + npc * (8 + 4 + 1 + 1) + 32
    if nta_L:
        b += npc * (nta_L + 1) * 8 + npc * 4 + npc * nta_L * 4 + 64
    return b


def rows_per_thread(npc, block):
    return -(-npc // block)


def _props():
    import torch
    return torch.cuda.get_device_properties(0)


def _sm():
    return _props().multi_processor_count


@pytest.fixture(scope="module")
def gpu():
    from volcano_b200 import engine
    engine.init(0)
    return engine


@contextlib.contextmanager
def tunables(**opts):
    """Diagnostic switches of libvcalloc (vc_debug_option) for the body only; every one is reset to 0 afterwards."""
    from volcano_b200 import engine
    try:
        for k, v in opts.items():
            engine.debug_option(k, v)
        yield
    finally:
        for k in opts:
            engine.debug_option(k, 0)


def _host_threads():
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(16, n))


def _assert_same(a, b):
    """Decisions (task, node, kind, visit, fp64 score bit for bit), visits, fit errors, allocated hypernodes."""
    assert len(a.visits) == len(b.visits), (len(a.visits), len(b.visits))
    for f in ("job", "outcome", "n_ops", "first_op"):
        assert np.array_equal(a.visits[f], b.visits[f]), f
    assert len(a.decisions) == len(b.decisions), (len(a.decisions), len(b.decisions))
    for f in ("task", "node", "kind", "visit"):
        if not np.array_equal(a.decisions[f], b.decisions[f]):
            i = int(np.nonzero(a.decisions[f] != b.decisions[f])[0][0])
            raise AssertionError(f"decision {i} differs in {f}: {a.decisions[i]} vs {b.decisions[i]}")
    if not np.array_equal(a.decisions["score"], b.decisions["score"]):
        i = int(np.nonzero(a.decisions["score"] != b.decisions["score"])[0][0])
        raise AssertionError(f"decision {i}: score {a.decisions['score'][i]!r} vs {b.decisions['score'][i]!r}")
    assert np.array_equal(a.fit_errors, b.fit_errors)
    if b.job_allocated_hypernodes is not None:
        assert a.job_allocated_hypernodes is not None
        assert np.array_equal(a.job_allocated_hypernodes, b.job_allocated_hypernodes)


def _assert_same_evict(a, b):
    assert (a is None) == (b is None)
    if a is None:
        return
    assert np.array_equal(a.visits, b.visits), (a.visits, b.visits)
    for f in ("task", "node", "kind", "visit"):
        assert np.array_equal(a.decisions[f], b.decisions[f]), f


def _assert_cycle(res, ref):
    """Every action of the cycle: allocate, then backfill / preempt / reclaim where the session has them."""
    _assert_same(res, ref)
    assert (res.backfill is None) == (ref.backfill is None)
    if ref.backfill is not None:
        _assert_same(res.backfill, ref.backfill)
    _assert_same_evict(res.preempt, ref.preempt)
    _assert_same_evict(res.reclaim, ref.reclaim)


def _small(name, n_nodes, n_tasks, **kw):
    from volcano_b200 import synth
    return dataclasses.replace(synth.CONFIGS["small"], name=name, n_nodes=n_nodes, n_tasks=n_tasks, **kw)


def _sampling(snap, pct=30, start=None):
    snap.conf.percentage_nodes_to_find = pct
    snap.conf.last_processed_node_index = start if start is not None else snap.N // 3 + 7
    return snap


def _oracle_sampled(snap):
    """Oracle allocate with feasible-node sampling (single-worker reading) and its util.lastProcessedNodeIndex."""
    from oracle import pyoracle
    from oracle.pyoracle import OracleSession
    from volcano_b200.uthelper import AllocateResult
    o = OracleSession(snap, threads=1)
    ref = AllocateResult(*o.allocate())
    last = pyoracle.lib().vco_last_processed_node_index(o.h)
    o.close()
    return ref, last


def _generator(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "tools", f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ---------------------------------------------------------------------------------------------------------------------
# the helper against the numbers DESIGN.md states (no GPU needed)
# ---------------------------------------------------------------------------------------------------------------------
def test_expected_geometry_matches_design():
    assert expected_geometry(10_000, 148, True) == (79, 128, 256)  # 79 x 128 on the incremental kernel
    assert expected_geometry(10_000, 148, False)[:2] == (105, 96)  # the general kernel keeps 96 nodes per CTA
    G, npc, block = expected_geometry(50_000, 148, True)
    assert npc == 352 and rows_per_thread(npc, block) == 2
    # the regimes the cases below are named after
    assert expected_geometry(4_500, 148, True)[0] == 141
    assert expected_geometry(6_000, 148, True)[1] == 64
    assert expected_geometry(8_191, 148, True)[1] == 64 and expected_geometry(8_192, 148, True)[1] == 128
    assert expected_geometry(18_000, 148, True)[:2] == (141, 128)
    assert rows_per_thread(*expected_geometry(40_000, 148, True)[1:]) == 2
    assert expected_geometry(700, 148, True, ctas=1) == (1, 704, 256)
    assert expected_geometry(700, 148, True, threads=160) == (22, 32, 160)
    # 1 200 nodes on one CTA: five node rows, more than feasible-node sampling supports
    assert rows_per_thread(*expected_geometry(1_200, 148, True, ctas=1)[1:]) == 5
    # FUT rows at 704 nodes per CTA do not fit a B200 CTA (227 KB); the plain rows do
    assert commit_smem(704, 1, 8, 3, True, True) > 232_448 > commit_smem(704, 1, 8, 3, True, False)


def test_wide_resource_vector_over_the_limit_is_refused():
    """R = 17 dimensions (cpu, memory, pods and 14 named scalars): encode_cluster refuses it by name."""
    tc = _wide_cluster(17, 1, "allocate")
    with pytest.raises(ValueError, match="17 resource dimensions"):
        tc.RegisterSession(_wide_tiers(17, "allocate"))


# ---------------------------------------------------------------------------------------------------------------------
# 1. node-count regimes at the default geometry
# ---------------------------------------------------------------------------------------------------------------------
REGIMES = [(1, "one_node"), (31, "one_warp_short"), (33, "last_cta_one_node"), (63, "two_warps_short"),
           (65, "mask_word_plus_one"), (127, "four_warps_short"), (129, "last_cta_one_node_5"),
           (4_500, "G_over_128_npc32"), (6_000, "npc64"), (8_191, "npc64_below_switch"), (8_192, "npc128_at_switch"),
           (18_000, "G_over_128_npc128"), (40_000, "two_rows_per_thread")]
MODES = ["plain", "fut_soft"]


def _regime_cfg(N, mode):
    T = min(4_000, max(64, 6 * N))
    extra = dict(releasing_frac=0.4, soft_taint_p=0.05, utilisation=0.9, min_util=0.5) if mode == "fut_soft" else {}
    return _small(f"regime{N}_{mode}", N, T, **extra)


def _check_regime(N, regime, fast, sm, rows=None):
    G, npc, block = expected_geometry(N, sm, fast)
    if regime.startswith("last_cta_one_node"):
        assert N - (G - 1) * npc == 1 and G >= 2
    elif regime == "G_over_128_npc32":
        assert G > 128 and npc == 32
    elif regime == "npc64" or regime == "npc64_below_switch":
        assert npc == 64
    elif regime == "npc128_at_switch":
        assert npc == 128 and N == 64 * 128
    elif regime == "G_over_128_npc128":
        assert G > 128 and npc == 128
    elif regime == "two_rows_per_thread":
        assert rows_per_thread(npc, block) == 2
    return G, npc, block


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("N,regime", REGIMES, ids=[f"{n}-{r}" for n, r in REGIMES])
def test_node_count_regimes_vs_oracle(N, regime, mode, gpu, oracle_engine):
    from volcano_b200.synth import make_snapshot
    snap = make_snapshot(_regime_cfg(N, mode), 17 + N % 97)
    res = gpu.gpu_engine(snap)
    assert res.stats["commit_kernel"] == VC_KERNEL_INCREMENTAL, res.stats
    _check_regime(N, regime, True, _sm())
    ref = oracle_engine(snap, threads=_host_threads())
    _assert_same(res, ref)
    assert len(ref.decisions) > 0 or N == 1  # (one node holds none of the gangs)
    if mode == "fut_soft":  # the <FUT, SOFT> instance: Releasing rows and PreferNoSchedule taints present
        assert snap.n_releasing.any() and snap.n_taint_soft.any()


SAMPLED_REGIMES = [(4_500, "G_over_128_npc32"), (40_000, "two_rows_per_thread")]


@pytest.mark.gpu
@pytest.mark.parametrize("N,regime", SAMPLED_REGIMES, ids=[f"{n}-{r}" for n, r in SAMPLED_REGIMES])
def test_node_count_regimes_sampling_vs_oracle(N, regime, gpu):
    """Feasible-node sampling (percentage-nodes-to-find 30, rotating start index != 0) on the SAMP instance."""
    from volcano_b200.synth import make_snapshot
    snap = _sampling(make_snapshot(_regime_cfg(N, "plain"), 5 + N % 89))
    res = gpu.gpu_engine(snap)
    assert res.stats["commit_kernel"] == VC_KERNEL_INCREMENTAL, res.stats
    _check_regime(N, regime, True, _sm())
    ref, last = _oracle_sampled(snap)
    _assert_same(res, ref)
    assert res.stats["last_processed_node_index"] == last
    assert len(ref.decisions) > 0


# ---------------------------------------------------------------------------------------------------------------------
# 2. cfg4_flat at full size (50k nodes x 1M tasks, two node rows per thread)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cfg4_flat_full_size(gpu):
    """BASELINE config 4's shape without the topology plugin, on the incremental kernel: a rerun gives the same result,
    no node is over-committed, gang minimum holds, and every 100th decision re-derived by the oracle on the state the
    GPU's decisions reached is the same (node, fp64 score)."""
    from oracle.pyoracle import OracleSession
    from volcano_b200.synth import make_snapshot
    snap = make_snapshot("cfg4_flat")
    G, npc, block = expected_geometry(snap.N, _sm(), True)
    assert rows_per_thread(npc, block) == 2
    e = gpu.Engine(snap)
    e.upload()
    r1 = e.allocate()
    r2 = e.allocate()
    e.close()
    assert r1.stats["commit_kernel"] == VC_KERNEL_INCREMENTAL, r1.stats
    assert np.array_equal(r1.decisions, r2.decisions) and np.array_equal(r1.visits, r2.visits)
    dec = r1.decisions
    assert len(dec) > 500_000
    assert len(np.unique(dec["task"])) == len(dec)
    used = snap.n_used.copy()
    np.add.at(used.T, dec["node"], snap.t_resreq.T[dec["task"]])
    assert (used <= snap.n_allocatable + 0.1).all()
    committed = r1.visits["outcome"][dec["visit"]] == 0
    per_job = np.bincount(snap.t_job[dec["task"][committed]], minlength=snap.J)
    jobs_committed = np.unique(r1.visits["job"][r1.visits["outcome"] == 0])
    assert (per_job[jobs_committed] >= snap.j_min_available[jobs_committed]).all()
    o = OracleSession(snap, threads=_host_threads())
    bad, first, checked = o.replay_check(r1.decisions, r1.visits, 100, 41)
    o.close()
    assert checked >= len(dec) // 100 - 1
    assert bad == 0, f"{bad} of {checked} sampled decisions differ, first at index {first}"


# ---------------------------------------------------------------------------------------------------------------------
# 3. forced geometries: no switch changes a result
# ---------------------------------------------------------------------------------------------------------------------
INSTANCES = ["small", "small_fut_soft", "small_roles", "small_bf", "tiny_topo", "small_sampling"]
SWITCHES = ([("VC_COMMIT_CTAS", c) for c in (1, 2, 3, 7)] + [("VC_COMMIT_THREADS", t) for t in (128, 160, 256)] +
            [("VC_RUN_MAX", r) for r in (1, 2, 5, 32)])


def _instance(name):
    from volcano_b200.synth import make_snapshot
    if name == "small_sampling":
        return _sampling(make_snapshot("small", 3), 30, 333)
    return make_snapshot(name, None)


def _expected_smem(snap, fast, G, npc):
    """Shared memory of the commit CTA of `snap` at (G, npc), and whether the device holds it."""
    sampling = snap.conf.percentage_nodes_to_find < 100
    topo = snap.hn_job_soft is not None and bool(snap.hn_job_soft.any())
    future = bool(snap.n_releasing.any() or snap.n_pipelined.any()) or topo or sampling
    nta_L = snap.hn_member.shape[0] if not fast and snap.hn_member is not None else 0  # hypernode tables (upper bound)
    b = commit_smem(npc, G, snap.R, snap.K, fast, future, nta_L)
    return b, b <= _props().shared_memory_per_block_optin


@pytest.fixture(scope="module")
def instance_refs(oracle_engine):
    """Per instance: the oracle's result (and lastProcessedNodeIndex under sampling) and the commit kernel that serves
    it on the default geometry. The switches touch neither, so each is computed once."""
    from volcano_b200 import engine
    cache = {}

    def get(name):
        if name not in cache:
            snap = _instance(name)
            ref, last = _oracle_sampled(snap) if name == "small_sampling" else (oracle_engine(snap, threads=_host_threads()), None)
            fast = engine.gpu_engine(snap).stats["commit_kernel"] == VC_KERNEL_INCREMENTAL
            cache[name] = (ref, last, fast)
        return cache[name]
    return get


FORCED = [(s, v, 0) for s, v in SWITCHES] + [("VC_COMMIT_CTAS", c, 1) for c in (0, 1, 2, 3, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("switch,value,generic", FORCED,
                         ids=[f"{s}={v}" + ("+generic" if g else "") for s, v, g in FORCED])
@pytest.mark.parametrize("name", INSTANCES)
def test_forced_geometry_vs_oracle(name, switch, value, generic, gpu, instance_refs):
    """Every instance under every switch equals the oracle; a geometry whose CTA would not fit the device's shared memory
    is refused by the library (VC_EUNSUPPORTED) before any launch."""
    from volcano_b200.abi import VC_EUNSUPPORTED
    ref, last, fast = instance_refs(name)
    fast = fast and not generic
    snap = _instance(name)
    G, npc, block = expected_geometry(snap.N, _sm(), fast, ctas=value if switch == "VC_COMMIT_CTAS" else 0,
                                      threads=value if switch == "VC_COMMIT_THREADS" else 0)
    if switch == "VC_COMMIT_CTAS" and value == 1 and snap.N == 700:
        assert (npc, rows_per_thread(npc, block)) == (704, 3)  # three node rows per thread
    smem, fits = _expected_smem(snap, fast, G, npc)
    opts = {switch: value, "VC_COMMIT_GENERIC": generic}
    if not fits:
        with tunables(**opts), pytest.raises(gpu.VcError) as ei:
            gpu.gpu_engine(snap)
        assert ei.value.code == VC_EUNSUPPORTED and "shared memory" in str(ei.value), (smem, ei.value)
        return
    with tunables(**opts):
        res = gpu.gpu_engine(snap)
    assert res.stats["commit_kernel"] == (VC_KERNEL_INCREMENTAL if fast else VC_KERNEL_GENERAL), res.stats
    _assert_cycle(res, ref)
    if last is not None:
        assert res.stats["last_processed_node_index"] == last


@pytest.mark.gpu
def test_sampling_refuses_more_than_four_node_rows(gpu):
    """Feasible-node sampling supports at most 4 node rows per CTA: 1 200 nodes on one CTA (1 216 nodes, 5 rows) is
    refused by name, for an allocate + backfill cycle and for a backfill-only one."""
    from volcano_b200.abi import VC_EUNSUPPORTED
    from volcano_b200.synth import make_snapshot
    cfg = _small("samp_rows", 1_200, 600, n_besteffort=200)
    G, npc, block = expected_geometry(1_200, _sm(), True, ctas=1)
    assert rows_per_thread(npc, block) == 5
    for actions in (("allocate", "backfill"), ("backfill",)):
        snap = _sampling(make_snapshot(cfg, 2), 30, 17)
        snap.actions = actions
        assert snap.B > 0
        with tunables(VC_COMMIT_CTAS=1):
            e = gpu.Engine(snap)
            try:
                with pytest.raises(gpu.VcError) as ei:
                    e.upload()
                    e.allocate() if "allocate" in actions else e.backfill()
            finally:
                e.close()
        assert ei.value.code == VC_EUNSUPPORTED and "node rows per CTA" in str(ei.value), ei.value
    # the same session on the default geometry runs
    snap = _sampling(make_snapshot(cfg, 2), 30, 17)
    assert len(gpu.gpu_engine(snap).decisions) > 0


@pytest.mark.gpu
def test_commit_kernel_not_co_resident_is_refused(gpu):
    """More CTAs than the device can hold at once (one node warp each, 256 threads: at most 8 per SM) cannot run the
    cooperative commit kernel: refused by name before the launch."""
    from volcano_b200.abi import VC_EUNSUPPORTED
    from volcano_b200.synth import make_snapshot
    sm = _sm()
    ctas = 8 * sm + 8
    N = 32 * ctas
    assert ctas <= 2048
    G, npc, block = expected_geometry(N, sm, True, ctas=ctas)
    assert G == ctas and npc == 32 and block == 256
    snap = make_snapshot(_small("coresident", N, 200), 4)
    with tunables(VC_COMMIT_CTAS=ctas):
        with pytest.raises(gpu.VcError) as ei:
            gpu.gpu_engine(snap)
    assert ei.value.code == VC_EUNSUPPORTED and "co-resident" in str(ei.value), ei.value


# ---------------------------------------------------------------------------------------------------------------------
# 4. randomised clusters on many CTAs
# ---------------------------------------------------------------------------------------------------------------------
FUZZ_BLOCKS = [("big", {}), ("big", {"VC_COMMIT_CTAS": 1}), ("plain", {"VC_COMMIT_THREADS": 128})]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,opts", FUZZ_BLOCKS, ids=["big-default", "big-ctas1", "plain-threads128"])
def test_random_clusters_many_ctas(kind, opts, gpu, oracle_engine):
    """tools/fuzz_api.py clusters (every feature): 40-400 nodes on many CTAs and on one CTA (up to two node rows per
    thread), and the small ones on 128-thread blocks. A session whose CTA would not fit the device's shared memory on one CTA is
    refused by name; every other one equals the oracle."""
    gen = _generator("fuzz_api")
    seeds = range(7000, 7030) if kind == "big" else range(7100, 7140)
    checked = refused = 0
    for seed in seeds:
        tc, tiers, actions = gen.make_case(seed, big=(kind == "big"))
        if not tiers:
            continue
        if not gen.backfill_supported(tiers, tc.conf_kw):
            actions = tuple(a for a in actions if a != "backfill")
        snap = tc.RegisterSession(tiers, actions=actions, **tc.conf_kw)
        if snap.T == 0 or snap.N == 0:
            continue
        ref = oracle_engine(snap)
        try:
            with tunables(**opts):
                res = gpu.gpu_engine(snap)
        except gpu.VcError as e:
            from volcano_b200.abi import VC_EUNSUPPORTED
            assert opts.get("VC_COMMIT_CTAS") == 1 and e.code == VC_EUNSUPPORTED and "shared memory" in str(e), (seed, e)
            refused += 1
            continue
        try:
            _assert_cycle(res, ref)
        except AssertionError as e:
            raise AssertionError(f"seed {seed}: {e}") from e
        checked += 1
    assert checked >= 20 and refused <= checked // 2, (checked, refused)


# ---------------------------------------------------------------------------------------------------------------------
# 5. dense pass (K1) shapes
# ---------------------------------------------------------------------------------------------------------------------
DENSE = [("odd_701_plain_expand", 701, 2_000, 0, {}), ("n63", 63, 400, 0, {}), ("n64", 64, 400, 0, {}),
         ("n65", 65, 400, 0, {}), ("n129", 129, 800, 0, {}), ("even_700_expand_plain", 700, 2_000, 0, {"VC_EXPAND_PLAIN": 1}),
         ("chunk128", 700, 2_000, 0, {"VC_EXPAND_CHUNK": 128}), ("rows1", 700, 2_000, 0, {"VC_EXPAND_ROWS": 1}),
         ("rows3", 700, 2_000, 0, {"VC_EXPAND_ROWS": 3}), ("rows64", 700, 2_000, 0, {"VC_EXPAND_ROWS": 64}),
         ("bulk_two_chunks_8200", 8_200, 300, 0, {}), ("hetero", 500, 1_500, 1_000, {})]


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,T,hetero,opts", DENSE, ids=[d[0] for d in DENSE])
def test_score_matrix_shapes_vs_oracle(name, N, T, hetero, opts, gpu):
    from oracle.pyoracle import OracleSession
    from volcano_b200.synth import make_snapshot
    snap = make_snapshot(_small(f"dense_{name}", N, T, hetero=hetero), 9 + N)
    with tunables(**opts):
        e = gpu.Engine(snap)
        try:
            e.upload()
            mask, score, bs, bn = e.score_matrix()
        finally:
            e.close()
    o = OracleSession(snap)
    omask, oscore, obs, obn = o.score_matrix()
    o.close()
    assert mask.any()
    assert np.array_equal(mask, omask)
    assert np.array_equal(bn, obn)
    assert np.array_equal(bs, obs)
    assert np.array_equal(score, oscore), "scores are expected to be bit-identical"


# ---------------------------------------------------------------------------------------------------------------------
# 6. wide resource vectors (R > 8)
# ---------------------------------------------------------------------------------------------------------------------
def _scalars(R):
    # sort after "pods": the highest dimension is a named scalar some pods request
    return [f"vendor.io/r{i:02d}" for i in range(R - 3)]


def _wide_cluster(R, seed, action):
    """An API-level cluster with R dimensions: cpu, memory, pods and R-3 named scalars on every node. Pods request
    random subsets of the scalars (the top one often); for preempt / reclaim the nodes are filled with running pods of
    low-priority / over-used jobs and higher-priority / starving jobs wait."""
    from volcano_b200.api import BuildNode, BuildPod, BuildPodGroup, BuildQueue, BuildResourceList
    from volcano_b200.uthelper import TestCommonStruct
    rnd = random.Random(seed * 7919 + R)
    names = _scalars(R)
    top = names[-1]
    n_nodes = 24 if action == "allocate" else 8
    nodes = []
    for i in range(n_nodes):
        sc = [(s, str(rnd.choice([4, 8, 16]))) for s in names]
        nodes.append(BuildNode(f"n{i:02d}", BuildResourceList(str(rnd.choice([8, 16])), rnd.choice(["16Gi", "32Gi"]),
                                                              ("pods", "20"), *sc)))

    def req():
        pick = [s for s in names if rnd.random() < 0.3]
        if rnd.random() < 0.6:
            pick.append(top)
        return BuildResourceList(rnd.choice(["500m", "1", "2"]), rnd.choice(["1Gi", "2Gi"]),
                                 *[(s, str(rnd.choice([1, 2, 3]))) for s in sorted(set(pick))])

    cap = BuildResourceList("200", "400Gi", *[(s, "300") for s in names[-3:]])
    queues = [BuildQueue("q0", 1, cap), BuildQueue("q1", 2, None)]
    queues[1].guarantee = BuildResourceList("4", "8Gi", (top, "6"))
    pgs, pods = [], []
    if action == "allocate":
        for j in range(14):
            size = rnd.choice([1, 2, 4, 6])
            pgs.append(BuildPodGroup(f"pg{j}", "ns", f"q{j % 2}", rnd.choice([1, size])))
            for k in range(size):
                pods.append(BuildPod("ns", f"j{j}-{k}", "", "Pending", req(), f"pg{j}"))
            if j % 5 == 0:  # BestEffort pods for the backfill action
                pods.append(BuildPod("ns", f"j{j}-be", "", "Pending", {}, f"pg{j}"))
    else:
        # running pods fill the nodes on the top scalar; preempt: one queue, low-priority victims;
        # reclaim: q0 holds everything, q1 starves
        for j in range(6):
            pg = BuildPodGroup(f"run{j}", "ns", "q0", 1, phase="Running")
            pg.priority = 1
            pgs.append(pg)
        for i, n in enumerate(nodes):
            left = int(n.allocatable[top])
            k = 0
            while left > 0:
                r = req()
                r[top] = str(min(left, rnd.choice([2, 4])))
                left -= int(r[top])
                p = BuildPod("ns", f"run-{i}-{k}", n.name, "Running", r, f"run{(i + k) % 6}",
                             {"volcano.sh/preemptable": "true"})
                pods.append(p)
                k += 1
        wq = "q0" if action == "preempt" else "q1"
        for j in range(4):
            pg = BuildPodGroup(f"want{j}", "ns", wq, 1)
            pg.priority = 100
            pgs.append(pg)
            for k in range(rnd.choice([1, 2])):
                r = req()
                r[top] = str(rnd.choice([2, 3]))
                pods.append(BuildPod("ns", f"want{j}-{k}", "", "Pending", r, f"want{j}"))
    return TestCommonStruct(Name=f"wide{R}-{action}-{seed}", Nodes=nodes, Pods=pods, PodGroups=pgs, Queues=queues)


def _wide_tiers(R, action):
    from volcano_b200.snapshot import PluginOption
    names = _scalars(R)
    hi = names[-3:]
    bp = {"binpack.weight": 5, "binpack.cpu": 2, "binpack.memory": 1, "binpack.resources": ",".join(hi)}
    bp.update({f"binpack.resources.{s}": 3 + i for i, s in enumerate(hi)})
    scorers = [PluginOption.defaults("predicates"), PluginOption.defaults("nodeorder"), PluginOption.defaults("binpack", bp)]
    if action == "allocate":
        return [[PluginOption.defaults("priority"), PluginOption.defaults("gang")],
                [PluginOption.defaults("drf"), PluginOption.defaults("proportion")] + scorers]
    if action == "preempt":
        return [[PluginOption.make("conformance", EnabledPreemptable=True),
                 PluginOption.make("gang", EnabledPreemptable=True, EnabledJobPipelined=True, EnabledJobStarving=True),
                 PluginOption.make("priority", EnabledTaskOrder=True, EnabledJobOrder=True, EnabledPreemptable=True,
                                   EnabledJobPipelined=True, EnabledJobStarving=True),
                 PluginOption.make("proportion", EnabledOverused=True, EnabledAllocatable=True, EnabledQueueOrder=True)],
                scorers]
    return [[PluginOption.make("conformance", EnabledReclaimable=True),
             PluginOption.make("gang", EnabledReclaimable=True, EnabledJobStarving=True),
             PluginOption.make("proportion", EnabledReclaimable=True, EnabledQueueOrder=True, EnablePreemptive=True),
             PluginOption.make("priority", EnabledReclaimable=True, EnabledJobOrder=True, EnabledTaskOrder=True)],
            scorers]


WIDE = [(R, a) for a in ("allocate", "allocate_backfill", "preempt", "reclaim") for R in (9, 12, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("R,action", WIDE, ids=[f"R{r}-{a}" for r, a in WIDE])
def test_wide_resource_vectors_vs_oracle(R, action, gpu, oracle_engine):
    """More than 8 dimensions: the general commit kernel (the incremental one holds R <= 8), the dense pass, backfill and
    the evict ranking (k_evict_rank<16, 16>) against the oracle, with binpack weights and queue capability / guarantee
    on the top dimensions."""
    kind = action.split("_")[0]
    actions = {"allocate": ("allocate",), "allocate_backfill": ("allocate", "backfill"), "preempt": ("preempt",),
               "reclaim": ("reclaim",)}[action]
    checked = ops = 0
    for seed in range(3):
        tc = _wide_cluster(R, seed, kind)
        snap = tc.RegisterSession(_wide_tiers(R, kind), actions=actions)
        assert snap.R == R
        top_req = snap.t_resreq[R - 1]
        assert (top_req > 0).any()
        if kind == "allocate":
            assert (top_req == 0).any()  # the top dimension is requested by some pods only (the req_has bits)
        res = gpu.gpu_engine(snap)
        ref = oracle_engine(snap)
        if kind == "allocate":
            assert res.stats["commit_kernel"] == VC_KERNEL_GENERAL, res.stats
            assert len(ref.decisions) > 0
        if action == "allocate_backfill":
            assert ref.backfill is not None and len(ref.backfill.decisions) > 0
        _assert_cycle(res, ref)
        for r in (ref.preempt, ref.reclaim):
            if r is not None:
                ops += int((r.decisions["kind"] == 2).sum())
        checked += 1
    if kind in ("preempt", "reclaim"):
        assert ops > 0  # evictions happened


# ---------------------------------------------------------------------------------------------------------------------
# 7. large preempt / reclaim: k_evict_pick_big (more than 25 600 nodes)
# ---------------------------------------------------------------------------------------------------------------------
def _big_evict_cluster(N, n_pending, action, seed=5):
    """N full nodes (one preemptable running pod fills each), low-priority jobs of queue q0 on them, and `n_pending`
    higher-priority gangs (minAvailable = size, so a job stays starving until every pod has a place) waiting in q0
    (preempt: the only queue, never over its share) or in q1 (reclaim). make_cfg5 at this size leaves tens of thousands
    of pending tasks, which takes the oracle minutes; this cluster keeps the pick kernel's candidate list at N nodes
    with a few dozen preemptors."""
    from volcano_b200.api import BuildNode, BuildPod, BuildPodGroup, BuildQueue, BuildResourceList
    from volcano_b200.uthelper import TestCommonStruct
    rnd = random.Random(seed)
    nodes, pods, pgs = [], [], []
    for j in range(64):
        pg = BuildPodGroup(f"run{j}", "ns", "q0", 1, phase="Running")
        pg.priority = 1
        pgs.append(pg)
    for i in range(N):
        cpu = rnd.choice([4, 8])
        nodes.append(BuildNode(f"n{i:05d}", BuildResourceList(str(cpu), f"{2 * cpu}Gi", ("pods", "10"))))
        pods.append(BuildPod("ns", f"run-{i}", f"n{i:05d}", "Running", BuildResourceList(str(cpu), rnd.choice(["2Gi", "4Gi"])),
                             f"run{i % 64}", {"volcano.sh/preemptable": "true"}))
    q = "q0" if action == "preempt" else "q1"
    for j in range(4):
        pg = BuildPodGroup(f"want{j}", "ns", q, n_pending // 4)
        pg.priority = 100
        pgs.append(pg)
        for k in range(n_pending // 4):
            pods.append(BuildPod("ns", f"want{j}-{k}", "", "Pending", BuildResourceList(rnd.choice(["1", "2", "3"]), "1Gi"),
                                 f"want{j}"))
    queues = [BuildQueue("q0", 1, None)] + ([BuildQueue("q1", 1, None)] if action == "reclaim" else [])
    return TestCommonStruct(Name=f"big-evict{N}", Nodes=nodes, Pods=pods, PodGroups=pgs, Queues=queues)


def _big_evict_tiers(action):
    from volcano_b200.snapshot import PluginOption
    scorers = [PluginOption.defaults("predicates"), PluginOption.defaults("nodeorder"),
               PluginOption.defaults("binpack", {"binpack.weight": 3, "binpack.cpu": 2})]
    return _wide_tiers(9, action)[:1] + [scorers]


@pytest.mark.gpu
@pytest.mark.parametrize("action", ["preempt", "reclaim"])
def test_large_evict_pick_vs_oracle(action, gpu, oracle_engine):
    """26 000 nodes: the pick kernel's candidate keys (N x 8 B) no longer fit shared memory, so k_evict_pick_big serves
    every hand-out. Allocate, then the action; every decision and statement against the oracle."""
    tc = _big_evict_cluster(26_000, 48, action)
    snap = tc.RegisterSession(_big_evict_tiers(action), actions=("allocate", action))
    assert snap.N * 8 > 200 * 1024
    res = gpu.gpu_engine(snap)
    ref = oracle_engine(snap, threads=_host_threads())
    _assert_cycle(res, ref)
    st = getattr(ref, action)
    assert (st.decisions["kind"] == 2).sum() > 10
