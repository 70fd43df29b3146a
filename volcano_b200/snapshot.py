"""Session snapshot in the structure-of-arrays layout of include/vcalloc.h.

`Snapshot` owns the numpy arrays (host memory) and hands ctypes views to the C ABI.
`encode_cluster` is the host-side mirror of what the reference does between
cache.Snapshot() (pkg/scheduler/cache/cache.go:1467-1576), framework.openSession
(pkg/scheduler/framework/session.go:166-282) and the plugins' OnSessionOpen bookkeeping —
i.e. exactly the marshalling the cgo shim performs in Go (INTEGRATION.md).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import re

import numpy as np

from . import abi
from .api import (HyperNode, Node, Pod, PodGroup, Queue, TASK_PRIORITY_ANNOTATION, allocated_status, get_task_role,
                  get_task_status, pod_index_under_task, quantity_milli, quantity_value, Taint, Toleration,
                  NodeSelectorRequirement, pod_critical, pod_preemptable)


# ---------------------------------------------------------------------------------------
# conf.SchedulerConfiguration (pkg/scheduler/conf/scheduler_conf.go:28-107)
# ---------------------------------------------------------------------------------------
@dataclass
class PluginOption:
    name: str
    enabled: int = 0  # OR of abi.VC_EN_*; 0 mirrors the reference's nil pointers in unit tests
    arguments: Dict[str, object] = field(default_factory=dict)

    @staticmethod
    def make(name: str, arguments: Optional[Dict[str, object]] = None, **enables: bool) -> "PluginOption":
        """PluginOption{Name: ..., EnabledJobOrder: &trueValue, ...}."""
        flags = 0
        for k, v in enables.items():
            if k.lower() in ("enabledhierarchy", "enablehierarchy") and v:
                # hierarchical drf (plugins/drf/drf.go:147-156, hdrf) orders queues by a tree the path does not model
                raise NotImplementedError("drf with enableHierarchy (hdrf) is outside the accelerated path")
            if k not in abi.ENABLE_FLAGS:
                # extension points that do not touch the allocate path (EnabledPreemptable, ...)
                continue
            if v:
                flags |= abi.ENABLE_FLAGS[k]
        return PluginOption(name=name, enabled=flags, arguments=dict(arguments or {}))

    @staticmethod
    def defaults(name: str, arguments: Optional[Dict[str, object]] = None) -> "PluginOption":
        """A YAML-configured plugin after ApplyPluginConfDefaults (plugins/defaults.go:29-55)."""
        return PluginOption(name=name, enabled=abi.VC_EN_ALL, arguments=dict(arguments or {}))


@dataclass
class SchedulerConf:
    tiers: List[List[PluginOption]]
    actions: Sequence[str] = ("allocate",)
    enable_predicate_error_cache: bool = True  # allocate.go:105-109
    percentage_nodes_to_find: int = 100        # parity mode (SURVEY §8c); reference default 0 = adaptive
    min_nodes_to_find: int = 100               # options.go:48-51
    min_percentage_nodes_to_find: int = 5
    last_processed_node_index: int = 0         # util.lastProcessedNodeIndex carried over from the previous cycle

    @staticmethod
    def default() -> "SchedulerConf":
        """DefaultSchedulerConf (pkg/scheduler/util.go:38-51) restricted to plugins on this path."""
        return SchedulerConf(
            tiers=[[PluginOption.defaults("priority"), PluginOption.defaults("gang")],
                   [PluginOption.defaults("drf"), PluginOption.defaults("predicates"),
                    PluginOption.defaults("proportion"), PluginOption.defaults("nodeorder")]],
            actions=("enqueue", "allocate", "backfill"))


def _get_int(args: Dict[str, object], key: str, default: int) -> int:
    """framework.Arguments.GetInt (framework/arguments.go:36-61): unparsable -> keep default."""
    if key not in args:
        return default
    try:
        return int(str(args[key]).strip())
    except ValueError:
        return default


def _get_bool(args: Dict[str, object], key: str, default: bool) -> bool:
    if key not in args:
        return default
    v = args[key]
    if isinstance(v, bool):
        return v
    s = str(v).strip().lower()
    if s in ("1", "t", "true"):
        return True
    if s in ("0", "f", "false"):
        return False
    return default


def build_conf(conf: SchedulerConf, dim_names: Sequence[str], kdim_names: Sequence[str]) -> abi.vc_conf:
    c = abi.vc_conf()
    opts = [(ti, p) for ti, tier in enumerate(conf.tiers) for p in tier]
    if len(opts) > abi.VC_MAX_PLUGINS:
        raise ValueError("too many plugins")
    c.n_plugins = len(opts)
    for i, (ti, p) in enumerate(opts):
        c.plugins[i].plugin = abi.PLUGIN_IDS.get(p.name, abi.VC_PLUGIN_OTHER)
        c.plugins[i].tier = ti
        c.plugins[i].enabled = p.enabled
    # binpack arguments (plugins/binpack/binpack.go:94-158)
    c.binpack_weight = 1
    for d in range(abi.VC_MAX_DIMS):
        c.binpack_dim_weight[d] = -1
    # nodeorder defaults (plugins/nodeorder/nodeorder.go:131-171)
    c.w_least, c.w_most, c.w_balanced, c.w_node_affinity, c.w_taint_toleration = 1, 0, 1, 2, 3
    c.predicates_enable = abi.VC_PRED_NODE_AFFINITY | abi.VC_PRED_TAINT_TOLERATION
    # network-topology-aware defaults (network_topology_aware.go:56-63)
    c.nta_weight, c.nta_normal_pod_enable, c.nta_fading = 1, 1, 0.8
    for d in range(abi.VC_MAX_DIMS):
        c.nta_dim_weight[d] = -1
    for d, name in enumerate(dim_names):
        if name in ("cpu", "memory"):
            c.nta_dim_weight[d] = 1
    for _, p in opts:
        a = p.arguments
        if p.name == "binpack":
            w = _get_int(a, "binpack.weight", 1)
            cpu = _get_int(a, "binpack.cpu", 1)
            mem = _get_int(a, "binpack.memory", 1)
            cpu = 1 if cpu < 0 else cpu
            mem = 1 if mem < 0 else mem
            weights: Dict[str, int] = {}
            for r in str(a.get("binpack.resources", "") or "").split(","):
                r = r.strip()
                if not r:
                    continue
                rw = _get_int(a, "binpack.resources." + r, 1)
                weights[r] = 1 if rw < 0 else rw
            weights["cpu"] = cpu
            weights["memory"] = mem
            c.binpack_weight = w
            for d, name in enumerate(dim_names):
                c.binpack_dim_weight[d] = weights.get(name, -1)
        elif p.name == "nodeorder":
            c.w_node_affinity = _get_int(a, "nodeaffinity.weight", 2)
            c.w_least = _get_int(a, "leastrequested.weight", 1)
            c.w_most = _get_int(a, "mostrequested.weight", 0)
            c.w_balanced = _get_int(a, "balancedresource.weight", 1)
            c.w_taint_toleration = _get_int(a, "tainttoleration.weight", 3)
        elif p.name == "network-topology-aware":  # getPriorityWeight / getNormalPodConfig :155-219
            def nonneg(v):
                return 1 if v < 0 else v
            c.nta_weight = nonneg(_get_int(a, "weight", 1))
            weights = {}
            for r in str(a.get("hypernode.binpack.resources", "") or "").split(","):
                r = r.strip()
                if r:
                    weights[r] = nonneg(_get_int(a, "hypernode.binpack.resources." + r, 1))
            weights["cpu"] = nonneg(_get_int(a, "hypernode.binpack.cpu", 1))      # getBinPackWeight: cpu / memory
            weights["memory"] = nonneg(_get_int(a, "hypernode.binpack.memory", 1))  # never come from the map
            for d, name in enumerate(dim_names):
                c.nta_dim_weight[d] = weights.get(name, -1)
            c.nta_normal_pod_enable = 1 if _get_bool(a, "hypernode.binpack.normal-pod.enable", True) else 0
            fading = a.get("hypernode.binpack.normal-pod.fading", 0.8)
            fading = float(fading) if isinstance(fading, (int, float)) and not isinstance(fading, bool) else 0.8
            c.nta_fading = 0.8 if fading < 0 else fading
        elif p.name == "predicates":
            en = 0
            if _get_bool(a, "predicate.NodeAffinityEnable", True):
                en |= abi.VC_PRED_NODE_AFFINITY
            if _get_bool(a, "predicate.TaintTolerationEnable", True):
                en |= abi.VC_PRED_TAINT_TOLERATION
            c.predicates_enable = en
    for k in range(abi.VC_MAX_KDIMS):
        c.kdim_dim[k] = dim_names.index(kdim_names[k]) if k < len(kdim_names) and kdim_names[k] in dim_names else -1
    c.enable_predicate_error_cache = 1 if conf.enable_predicate_error_cache else 0
    c.enqueue_action_enabled = 1 if "enqueue" in conf.actions else 0
    c.percentage_nodes_to_find = conf.percentage_nodes_to_find
    c.min_nodes_to_find = conf.min_nodes_to_find
    c.min_percentage_nodes_to_find = conf.min_percentage_nodes_to_find
    c.last_processed_node_index = conf.last_processed_node_index
    return c


# ---------------------------------------------------------------------------------------
# Snapshot: numpy SoA + ctypes views
# ---------------------------------------------------------------------------------------
def _ptr(a: Optional[np.ndarray], ctype):
    if a is None:
        return C.cast(None, C.POINTER(ctype))
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(ctype))


_F64, _I32, _I64, _U32, _U64, _U8 = C.c_double, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_uint8


class Snapshot:
    """All arrays are C-contiguous numpy arrays with the dtypes/shapes of include/vcalloc.h."""

    NODE_F = ("allocatable", "idle", "used", "releasing", "pipelined")
    NODE_K = ("k8s_allocatable", "k8s_requested", "k8s_nonzero_requested")

    def __init__(self, N, T, J, Q, C_, NR, R, K=3, Wl=1, Wt=1, Z=0, pods_dim=-1, B=0):
        self.N, self.T, self.J, self.Q, self.C, self.NR, self.R, self.K = N, T, J, Q, C_, NR, R, K
        self.B = B  # BestEffort pending tasks (the backfill action's tasks; not part of T)
        self.RT = 0  # tasks that occupy nodes (victim candidates of preempt / reclaim), see set_running
        self.t_flags = np.zeros(T, np.uint32)  # VC_TASK_* per pending task
        self.t_nominated = np.full(T, -1, np.int32)  # node index of Pod.Status.NominatedNodeName per pending task, -1 none
        self.Wl, self.Wt, self.Z, self.pods_dim = Wl, Wt, Z, pods_dim
        f8, i4, i8, u4, u8 = np.float64, np.int32, np.int64, np.uint32, np.uint64
        # nodes
        for n in self.NODE_F:
            setattr(self, "n_" + n, np.zeros((R, N), f8))
        for n in self.NODE_K:
            setattr(self, "n_" + n, np.zeros((K, N), f8))
        self.n_max_tasks = np.zeros(N, i4)
        self.n_pod_count = np.zeros(N, i4)
        self.n_label_bits = np.zeros((Wl, N), u8)
        self.n_taint_hard = np.zeros((Wt, N), u8)
        self.n_taint_soft = np.zeros((Wt, N), u8)
        self.n_flags = np.zeros(N, u4)
        self.n_revocable_zone = np.full(N, -1, i4)
        self.zone_active = np.zeros(max(Z, 1), np.uint8)
        # tasks (t_*: allocate's tasks; b_*: the BestEffort tasks of the backfill action, same fields)
        for pre, n in (("t_", T), ("b_", B)):
            setattr(self, pre + "resreq", np.zeros((R, n), f8))
            setattr(self, pre + "req_has", np.zeros(n, u4))
            setattr(self, pre + "k8s_req", np.zeros((K, n), f8))
            setattr(self, pre + "k8s_nonzero_req", np.zeros((K, n), f8))
            setattr(self, pre + "job", np.zeros(n, i4))
            setattr(self, pre + "klass", np.zeros(n, i4))
            setattr(self, pre + "role", np.zeros(n, i4))
            setattr(self, pre + "priority", np.ones(n, i4))
            setattr(self, pre + "pod_index", np.full(n, -1, i8))
            setattr(self, pre + "creation_ts", np.zeros(n, i8))
            setattr(self, pre + "uid_rank", np.arange(n, dtype=u4))
        # classes
        MT = abi.VC_MAX_TERMS
        self.c_selector = np.zeros((C_, Wl), u8)
        self.c_n_affinity = np.zeros(C_, i4)
        self.c_affinity = np.zeros((C_, MT, Wl), u8)
        self.c_tolerated_hard = np.zeros((C_, Wt), u8)
        self.c_tolerated_soft = np.zeros((C_, Wt), u8)
        self.c_n_preferred = np.zeros(C_, i4)
        self.c_preferred = np.zeros((C_, MT, Wl), u8)
        self.c_preferred_weight = np.zeros((C_, MT), i4)
        self.c_flags = np.zeros(C_, u4)
        # jobs
        self.j_queue = np.zeros(J, i4)
        self.j_min_available = np.zeros(J, i4)
        self.j_priority = np.zeros(J, i4)
        self.j_creation_ts = np.zeros(J, i8)
        self.j_uid_rank = np.arange(J, dtype=u4)
        self.j_flags = np.zeros(J, u4)
        self.j_n_tasks_total = np.zeros(J, i4)
        self.j_ready_num = np.zeros(J, i4)
        self.j_waiting_num = np.zeros(J, i4)
        self.j_pending_besteffort = np.zeros(J, i4)
        self.j_valid_num = np.zeros(J, i4)
        self.j_task_min_total = np.zeros(J, i4)
        self.j_role_off = np.zeros(J + 1, i4)
        self.j_allocated = np.zeros((R, J), f8)
        self.r_min = np.zeros(NR, i4)
        self.r_occupied = np.zeros(NR, i4)
        self.r_pipelined = np.zeros(NR, i4)
        self.r_pending_other = np.zeros(NR, i4)
        self.r_valid = np.zeros(NR, i4)
        self.r_flags = np.zeros(NR, u4)
        # queues
        self.q_weight = np.ones(Q, i4)
        self.q_priority = np.zeros(Q, i4)
        self.q_creation_ts = np.zeros(Q, i8)
        self.q_uid_rank = np.arange(Q, dtype=u4)
        self.q_flags = np.full(Q, abi.VC_QUEUE_OPEN, u4)
        self.q_capability = np.zeros((R, Q), f8)
        self.q_capability_has = np.zeros(Q, u4)
        self.q_guarantee = np.zeros((R, Q), f8)
        self.q_guarantee_has = np.zeros(Q, u4)
        self.q_allocated = np.zeros((R, Q), f8)
        self.q_request = np.zeros((R, Q), f8)
        self.q_request_has = np.zeros(Q, u4)
        self.q_allocated_has = np.zeros(Q, u4)
        self.conf: Optional[abi.vc_conf] = None
        self.actions: Sequence[str] = ("allocate",)  # the configured action list (which Action objects the host runs)
        # HyperNode tree (None: no HyperNode objects in the session)
        self.hn_names: List[str] = []
        self.hn_min_tier = 1
        self.hn_max_tier = 1
        self.hn_member: Optional[np.ndarray] = None  # int32 [L][N]
        self.hn_tier: Optional[np.ndarray] = None
        self.hn_parent: Optional[np.ndarray] = None
        self.hn_job_soft: Optional[np.ndarray] = None
        self.hn_job_allocated: Optional[np.ndarray] = None
        self.hn_job_placed_off: Optional[np.ndarray] = None
        self.hn_job_placed_node: Optional[np.ndarray] = None
        # names for humans / tests
        self.dim_names: List[str] = []
        self.node_names: List[str] = []
        self.task_keys: List[str] = []
        self.backfill_task_keys: List[str] = []
        self.job_names: List[str] = []
        self.queue_names: List[str] = []

    def topology(self) -> Optional[abi.vc_hypernodes]:
        if self.hn_member is None:
            return None
        return abi.vc_hypernodes(len(self.hn_names), self.hn_min_tier, self.hn_max_tier, _ptr(self.hn_member, _I32),
                                 _ptr(self.hn_tier, _I32), _ptr(self.hn_parent, _I32), _ptr(self.hn_job_soft, _U8),
                                 _ptr(self.hn_job_allocated, _I32), _ptr(self.hn_job_placed_off, _I32),
                                 _ptr(self.hn_job_placed_node, _I32))

    # ---- ctypes views ----------------------------------------------------------------
    def dims(self) -> abi.vc_dims:
        return abi.vc_dims(self.N, self.T, self.J, self.Q, self.C, self.NR, self.R, self.K, self.Wl, self.Wt,
                           self.Z, self.pods_dim)

    def nodes(self) -> abi.vc_nodes:
        return abi.vc_nodes(
            _ptr(self.n_allocatable, _F64), _ptr(self.n_idle, _F64), _ptr(self.n_used, _F64),
            _ptr(self.n_releasing, _F64), _ptr(self.n_pipelined, _F64), _ptr(self.n_k8s_allocatable, _F64),
            _ptr(self.n_k8s_requested, _F64), _ptr(self.n_k8s_nonzero_requested, _F64),
            _ptr(self.n_max_tasks, _I32), _ptr(self.n_pod_count, _I32), _ptr(self.n_label_bits, _U64),
            _ptr(self.n_taint_hard, _U64), _ptr(self.n_taint_soft, _U64), _ptr(self.n_flags, _U32),
            _ptr(self.n_revocable_zone, _I32), _ptr(self.zone_active, _U8))

    def tasks(self, pre: str = "t_") -> abi.vc_tasks:
        g = lambda name: getattr(self, pre + name)
        return abi.vc_tasks(
            _ptr(g("resreq"), _F64), _ptr(g("req_has"), _U32), _ptr(g("k8s_req"), _F64),
            _ptr(g("k8s_nonzero_req"), _F64), _ptr(g("job"), _I32), _ptr(g("klass"), _I32),
            _ptr(g("role"), _I32), _ptr(g("priority"), _I32), _ptr(g("pod_index"), _I64),
            _ptr(g("creation_ts"), _I64), _ptr(g("uid_rank"), _U32))

    def set_running(self, n: int):
        """Allocate the node.Tasks table (vc_running_tasks) for n occupying tasks."""
        f8, i4, i8, u4 = np.float64, np.int32, np.int64, np.uint32
        self.RT = n
        self.rt_node = np.zeros(n, i4); self.rt_job = np.full(n, -1, i4); self.rt_role = np.full(n, -1, i4)
        self.rt_priority = np.ones(n, i4); self.rt_pod_index = np.full(n, -1, i8); self.rt_creation_ts = np.zeros(n, i8)
        self.rt_uid_rank = np.arange(n, dtype=u4)
        self.rt_resreq = np.zeros((self.R, n), f8); self.rt_req_has = np.zeros(n, u4)
        self.rt_k8s_req = np.zeros((self.K, n), f8); self.rt_k8s_nonzero_req = np.zeros((self.K, n), f8)
        self.rt_flags = np.zeros(n, u4)
        self.running_task_keys = [""] * n

    def running_tasks(self) -> Optional[abi.vc_running_tasks]:
        """The argument of vc_snapshot_set_running, or None when no task occupies a node."""
        if getattr(self, "RT", 0) <= 0:
            return None
        return abi.vc_running_tasks(
            self.RT, _ptr(self.rt_node, _I32), _ptr(self.rt_job, _I32), _ptr(self.rt_role, _I32),
            _ptr(self.rt_priority, _I32), _ptr(self.rt_pod_index, _I64), _ptr(self.rt_creation_ts, _I64),
            _ptr(self.rt_uid_rank, _U32), _ptr(self.rt_resreq, _F64), _ptr(self.rt_req_has, _U32),
            _ptr(self.rt_k8s_req, _F64), _ptr(self.rt_k8s_nonzero_req, _F64), _ptr(self.rt_flags, _U32))

    def dump(self, path: str) -> None:
        """The session as a flat binary file a C program can feed to the C ABI (tools/cdriver/vcalloc_driver.c):
        magic "VCSNAP01", vc_dims, vc_conf, then the arrays of vc_nodes, vc_tasks, vc_classes, vc_jobs, vc_queues in the
        field order of include/vcalloc.h, each as uint64 byte count + raw little-endian bytes."""
        import ctypes as C
        g = lambda name: getattr(self, "t_" + name)
        arrays = [
            # vc_nodes
            self.n_allocatable, self.n_idle, self.n_used, self.n_releasing, self.n_pipelined, self.n_k8s_allocatable,
            self.n_k8s_requested, self.n_k8s_nonzero_requested, self.n_max_tasks, self.n_pod_count, self.n_label_bits,
            self.n_taint_hard, self.n_taint_soft, self.n_flags, self.n_revocable_zone, self.zone_active,
            # vc_tasks
            g("resreq"), g("req_has"), g("k8s_req"), g("k8s_nonzero_req"), g("job"), g("klass"), g("role"), g("priority"),
            g("pod_index"), g("creation_ts"), g("uid_rank"),
            # vc_classes
            self.c_selector, self.c_n_affinity, self.c_affinity, self.c_tolerated_hard, self.c_tolerated_soft,
            self.c_n_preferred, self.c_preferred, self.c_preferred_weight, self.c_flags,
            # vc_jobs
            self.j_queue, self.j_min_available, self.j_priority, self.j_creation_ts, self.j_uid_rank, self.j_flags,
            self.j_n_tasks_total, self.j_ready_num, self.j_waiting_num, self.j_pending_besteffort, self.j_valid_num,
            self.j_task_min_total, self.j_role_off, self.j_allocated, self.r_min, self.r_occupied, self.r_pipelined,
            self.r_pending_other, self.r_valid, self.r_flags,
            # vc_queues
            self.q_weight, self.q_priority, self.q_creation_ts, self.q_uid_rank, self.q_flags, self.q_capability,
            self.q_capability_has, self.q_guarantee, self.q_guarantee_has, self.q_allocated, self.q_request,
            self.q_request_has, self.q_allocated_has,
        ]
        with open(path, "wb") as f:
            f.write(b"VCSNAP01")
            f.write(bytes(self.dims()))
            f.write(bytes(self.conf))
            for a in arrays:
                b = np.ascontiguousarray(a).tobytes()
                f.write(np.uint64(len(b)).tobytes())
                f.write(b)

    def backfill_tasks(self) -> Optional[abi.vc_tasks]:
        """The argument of vc_snapshot_set_backfill, or None when the session has no BestEffort pending task."""
        return self.tasks("b_") if self.B > 0 else None

    def classes(self) -> abi.vc_classes:
        return abi.vc_classes(
            _ptr(self.c_selector, _U64), _ptr(self.c_n_affinity, _I32), _ptr(self.c_affinity, _U64),
            _ptr(self.c_tolerated_hard, _U64), _ptr(self.c_tolerated_soft, _U64), _ptr(self.c_n_preferred, _I32),
            _ptr(self.c_preferred, _U64), _ptr(self.c_preferred_weight, _I32), _ptr(self.c_flags, _U32))

    def jobs(self) -> abi.vc_jobs:
        return abi.vc_jobs(
            _ptr(self.j_queue, _I32), _ptr(self.j_min_available, _I32), _ptr(self.j_priority, _I32),
            _ptr(self.j_creation_ts, _I64), _ptr(self.j_uid_rank, _U32), _ptr(self.j_flags, _U32),
            _ptr(self.j_n_tasks_total, _I32), _ptr(self.j_ready_num, _I32), _ptr(self.j_waiting_num, _I32),
            _ptr(self.j_pending_besteffort, _I32), _ptr(self.j_valid_num, _I32), _ptr(self.j_task_min_total, _I32),
            _ptr(self.j_role_off, _I32), _ptr(self.j_allocated, _F64), _ptr(self.r_min, _I32),
            _ptr(self.r_occupied, _I32), _ptr(self.r_pipelined, _I32), _ptr(self.r_pending_other, _I32),
            _ptr(self.r_valid, _I32), _ptr(self.r_flags, _U32))

    def queues(self) -> abi.vc_queues:
        return abi.vc_queues(
            _ptr(self.q_weight, _I32), _ptr(self.q_priority, _I32), _ptr(self.q_creation_ts, _I64),
            _ptr(self.q_uid_rank, _U32), _ptr(self.q_flags, _U32), _ptr(self.q_capability, _F64),
            _ptr(self.q_capability_has, _U32), _ptr(self.q_guarantee, _F64), _ptr(self.q_guarantee_has, _U32),
            _ptr(self.q_allocated, _F64), _ptr(self.q_request, _F64), _ptr(self.q_request_has, _U32),
            _ptr(self.q_allocated_has, _U32))

    def input_bytes(self) -> int:
        """Bytes a full upload moves host->device."""
        tot = 0
        for k, v in self.__dict__.items():
            if isinstance(v, np.ndarray):
                tot += v.nbytes
        return tot


# ---------------------------------------------------------------------------------------
# cluster objects -> Snapshot
# ---------------------------------------------------------------------------------------
_K8S_DEFAULT_MILLI_CPU = 100           # schedutil.DefaultMilliCPURequest
_K8S_DEFAULT_MEMORY = 200 * 1024 * 1024  # schedutil.DefaultMemoryRequest
KDIM_NAMES = ("cpu", "memory", "nvidia.com/gpu")  # nodeorder.go:238-244


def _resource_vector(rl: Optional[Dict[str, str]], dim_names: Sequence[str]):
    """api.NewResource (api/resource_info.go:86-127) -> (values[R], has-mask)."""
    v = np.zeros(len(dim_names))
    has = 0
    for name, q in (rl or {}).items():
        if name == "cpu":
            v[0] += quantity_milli(q)
        elif name == "memory":
            v[1] += quantity_value(q)
        elif name.startswith("count/"):
            continue
        else:
            d = dim_names.index(name)
            v[d] += quantity_value(q) if name == "pods" else quantity_milli(q)
            has |= 1 << d
    return v, has


def _k8s_vector(rl: Optional[Dict[str, str]], nonzero: bool):
    out = np.zeros(len(KDIM_NAMES))
    rl = rl or {}
    for k, name in enumerate(KDIM_NAMES):
        if name in rl:
            out[k] = quantity_milli(rl[name]) if name == "cpu" else quantity_value(rl[name])
        elif nonzero and name == "cpu":
            out[k] = _K8S_DEFAULT_MILLI_CPU
        elif nonzero and name == "memory":
            out[k] = _K8S_DEFAULT_MEMORY
    return out


_RZ_RE = re.compile(r"(\d{1,2}):(\d{2})")


def parse_revocable_zone(rz_raw: str, now=None):
    """parseRevocableZone (plugins/tdm/tdm.go:88-116): "H:MM-H:MM" -> (start, end) datetimes of today's window;
    an end at or before the start rolls to tomorrow.  Raises ValueError on the inputs the reference rejects."""
    import datetime as _dt
    now = now or _dt.datetime.now()
    parts = rz_raw.strip().split("-")
    if len(parts) != 2:
        raise ValueError(f"revocable zone {rz_raw} format error")
    hm = []
    for v in parts:  # Go layout "15:04": one or two hour digits, exactly two minute digits
        m = _RZ_RE.fullmatch(v)
        if not m or int(m.group(1)) > 23 or int(m.group(2)) > 59:
            raise ValueError(f"parsing time {v!r}")
        hm.append((int(m.group(1)), int(m.group(2))))
    start = now.replace(hour=hm[0][0], minute=hm[0][1], second=0, microsecond=0)
    end = now.replace(hour=hm[1][0], minute=hm[1][1], second=0, microsecond=0)
    if hm[0] >= hm[1]:
        end += _dt.timedelta(days=1)
    return start, end


def tdm_zones_active(arguments: Dict[str, object], now=None) -> Dict[str, bool]:
    """availableRevocableZone (tdm.go:118-137) for every "tdm.revocable-zone.<name>" argument (tdm.go:65-77)."""
    import datetime as _dt
    now = now or _dt.datetime.now()
    out = {}
    for k, v in arguments.items():
        if not k.startswith("tdm.revocable-zone."):
            continue
        name = k[len("tdm.revocable-zone."):]
        try:
            start, end = parse_revocable_zone(str(v), now)
            out[name] = int(start.timestamp()) <= int(now.timestamp()) <= int(end.timestamp())
        except ValueError:
            out[name] = False
    return out


CLUSTER_TOP_HYPERNODE = "<cluster-top-hypernode>"  # framework.ClusterTopHyperNode


def encode_hypernodes(s: "Snapshot", hypernodes: Sequence[HyperNode], podgroups: Sequence[PodGroup] = (),
                      job_pods: Sequence[Sequence[Pod]] = ()) -> None:
    """ssn.HyperNodesSetByTier + ssn.RealNodesSet (framework/session.go:239-245) as a [tier level][node] table of
    hypernode indices, with the cluster top hypernode of addClusterTopHyperNode (:285-313) appended: its tier
    is one above the highest real tier and its RealNodesSet is the whole NodeList."""
    by_name = {h.name: h for h in hypernodes}
    nidx = {n: i for i, n in enumerate(s.node_names)}
    real: Dict[str, set] = {}

    def real_nodes(name, seen=()):
        if name in real:
            return real[name]
        out = set()
        for mname, mtype in by_name[name].members:
            if mtype == "Node":
                if mname in nidx:  # GetRealNodesByHyperNode keeps nodes of the snapshot only
                    out.add(nidx[mname])
            elif mname in by_name and mname not in seen:
                out |= real_nodes(mname, seen + (name,))
        real[name] = out
        return out

    top_tier = 1
    for h in hypernodes:
        real_nodes(h.name)
        top_tier = max(top_tier, h.tier + 1)
    names = sorted(by_name) + [CLUSTER_TOP_HYPERNODE]
    tiers = {h.name: h.tier for h in hypernodes}
    tiers[CLUSTER_TOP_HYPERNODE] = top_tier
    real[CLUSTER_TOP_HYPERNODE] = set(range(len(s.node_names)))
    s.hn_names = names
    s.hn_min_tier = min(tiers.values())
    s.hn_max_tier = top_tier
    L = s.hn_max_tier - s.hn_min_tier + 1
    if L > abi.VC_MAX_TIERS:
        raise ValueError("too many hypernode tiers")
    s.hn_member = np.full((L, len(s.node_names)), -1, np.int32)
    for hi, name in reversed(list(enumerate(names))):  # lowest name wins where sets of one tier overlap
        l = tiers[name] - s.hn_min_tier
        for n in real[name]:
            s.hn_member[l, n] = hi
    # HyperNodeInfo.Parent (api/hyper_node_info.go BuildHyperNodeCache; parentless ones hang under the cluster top)
    hidx = {name: i for i, name in enumerate(names)}
    s.hn_tier = np.array([tiers[n] for n in names], np.int32)
    s.hn_parent = np.full(len(names), -1, np.int32)
    for h in hypernodes:
        for mname, mtype in h.members:
            if mtype == "HyperNode" and mname in hidx:
                s.hn_parent[hidx[mname]] = hidx[h.name]
    for name in by_name:
        if s.hn_parent[hidx[name]] < 0:
            s.hn_parent[hidx[name]] = hidx[CLUSTER_TOP_HYPERNODE]
    # soft-mode topology jobs: subJob.AllocatedHyperNode at open (carried annotation, else recovered from the
    # nodes of the allocated tasks: lowest-tier hypernode holding all of them, framework/session.go:360-445)
    J = len(podgroups)
    s.hn_job_soft = np.zeros(J, np.uint8)
    s.hn_job_allocated = np.full(J, -1, np.int32)
    off, placed = [0], []
    for j, pg in enumerate(podgroups):
        nodes_j = [nidx[p.node_name] for p in job_pods[j] if p.node_name in nidx]
        placed.extend(nodes_j)
        off.append(len(placed))
        if pg.network_topology_mode != "soft":
            continue
        s.hn_job_soft[j] = 1
        alloc_nodes = [nidx[p.node_name] for p in job_pods[j]
                       if p.node_name in nidx and allocated_status(get_task_status(p))]
        if pg.allocated_hypernode in hidx and alloc_nodes:  # removeInvalidAllocatedHyperNode :317-356
            s.hn_job_allocated[j] = hidx[pg.allocated_hypernode]
        elif alloc_nodes:
            cands = [hi for hi, name in enumerate(names) if all(n in real[name] for n in alloc_nodes)]
            if cands:
                s.hn_job_allocated[j] = min(cands, key=lambda hi: (s.hn_tier[hi], names[hi]))
    s.hn_job_placed_off = np.array(off, np.int32)
    s.hn_job_placed_node = np.array(placed if placed else [0], np.int32)


def encode_cluster(nodes: Sequence[Node], pods: Sequence[Pod], podgroups: Sequence[PodGroup],
                   queues: Sequence[Queue], conf: SchedulerConf, tdm_zone_active: Optional[Dict[str, bool]] = None,
                   hypernodes: Optional[Sequence[HyperNode]] = None) -> Snapshot:
    # ---- dimensions: cpu, memory, then scalars sorted by name -------------------------------
    scalars = set()
    for n in nodes:
        scalars.update(k for k in n.allocatable if k not in ("cpu", "memory") and not k.startswith("count/"))
    for p in pods:
        scalars.update(k for k in p.requests if k not in ("cpu", "memory") and not k.startswith("count/"))
    for q in queues:
        for rl in (q.capability, q.guarantee):
            scalars.update(k for k in (rl or {}) if k not in ("cpu", "memory"))
    scalars.add("pods")  # every pod requests pods:1 (api/pod_info.go:119)
    dim_names = ["cpu", "memory"] + sorted(scalars)
    R = len(dim_names)
    if R > abi.VC_MAX_DIMS:
        raise ValueError(f"{R} resource dimensions ({', '.join(dim_names)}): the engine holds at most {abi.VC_MAX_DIMS}")
    pods_dim = dim_names.index("pods")

    # ---- jobs (JobID = ns/podgroup, api/job_info.go:156-164) -------------------------------
    qidx = {q.name: i for i, q in enumerate(queues)}
    job_ids = [f"{pg.namespace}/{pg.name}" for pg in podgroups]
    jidx = {jid: i for i, jid in enumerate(job_ids)}
    job_pods: List[List[Pod]] = [[] for _ in podgroups]
    for p in pods:
        jid = f"{p.namespace}/{p.group_name}"
        if jid in jidx:
            job_pods[jidx[jid]].append(p)

    def pod_req(p: Pod):
        v, has = _resource_vector(p.requests, dim_names)
        v[pods_dim] += 1
        has |= 1 << pods_dim
        return v, has

    def is_best_effort(v):  # Resource.IsEmpty ignoring pods (api/resource_info.go:240-255)
        return all(v[d] < 0.1 for d in range(R) if d != pods_dim)

    # ---- tasks in scope + role tables -------------------------------------------------------
    task_pods: List[Pod] = []
    task_job: List[int] = []
    bf_pods: List[Pod] = []  # Pending BestEffort pods: backfill's tasks (backfill.go:140-151)
    bf_job: List[int] = []
    role_rows: List[Dict[str, int]] = []  # per job: role name -> row
    role_tables = {k: [] for k in ("min", "occ", "pip", "pending_other", "valid", "flags")}
    role_off = [0]
    J = len(podgroups)
    snap_j = {k: np.zeros(J, np.int32) for k in ("ready", "waiting", "pbe", "valid", "ntasks", "tmt")}
    j_alloc = np.zeros((R, J))
    for j, pg in enumerate(podgroups):
        rows: Dict[str, int] = {}
        base = role_off[-1]
        tmm = pg.min_task_member or {}

        def row(role: str) -> int:
            if role not in rows:
                rows[role] = base + len(rows)
                role_tables["min"].append(int(tmm.get(role, 0)))
                for k in ("occ", "pip", "pending_other", "valid"):
                    role_tables[k].append(0)
                fl = (abi.VC_ROLE_EMPTY_NAME if role == "" else 0) | (abi.VC_ROLE_IN_MIN_MAP if role in tmm else 0)
                role_tables["flags"].append(fl)
            return rows[role]

        for role in tmm:
            row(role)
        snap_j["tmt"][j] = sum(int(v) for v in tmm.values())
        for p in job_pods[j]:
            st = get_task_status(p)
            v, _ = pod_req(p)
            r = row(get_task_role(p))
            snap_j["ntasks"][j] += 1
            be = is_best_effort(v)
            if allocated_status(st):
                j_alloc[:, j] += v
            if st in ("Bound", "Binding", "Running", "Allocated", "Succeeded"):
                snap_j["ready"][j] += 1
            if st == "Pipelined":
                snap_j["waiting"][j] += 1
                role_tables["pip"][r] += 1
            if allocated_status(st) or st == "Succeeded" or (st == "Pending" and be):
                role_tables["occ"][r] += 1
            if allocated_status(st) or st in ("Succeeded", "Pipelined", "Pending"):
                role_tables["valid"][r] += 1
                snap_j["valid"][j] += 1
            if st == "Pending":
                if be:
                    snap_j["pbe"][j] += 1
                    role_tables["pending_other"][r] += 1
                    bf_pods.append(p)
                    bf_job.append(j)
                else:
                    task_pods.append(p)
                    task_job.append(j)
        if len(rows) > abi.VC_MAX_JOB_ROLES:
            raise ValueError("too many roles in one job")
        role_rows.append(rows)
        role_off.append(base + len(rows))

    # ---- label requirements -> bits ---------------------------------------------------------
    req_bits: Dict[tuple, int] = {}

    def bit_of(req: NodeSelectorRequirement) -> int:
        k = req.ident()
        if k not in req_bits:
            req_bits[k] = len(req_bits)
        return req_bits[k]

    hard_taints: Dict[tuple, int] = {}
    soft_taints: Dict[tuple, int] = {}
    for n in nodes:
        for t in n.taints:
            d = soft_taints if t.effect == "PreferNoSchedule" else hard_taints
            d.setdefault((t.key, t.value, t.effect), len(d))
    zones: Dict[str, int] = {}
    for n in nodes:
        if n.revocable_zone:
            zones.setdefault(n.revocable_zone, len(zones))

    class_keys: Dict[tuple, int] = {}
    class_defs: List[dict] = []
    task_class: List[int] = []
    for p in task_pods + bf_pods:
        sel = tuple(sorted(bit_of(NodeSelectorRequirement(k, "In", (v,))) for k, v in p.node_selector.items()))
        aff = tuple(tuple(sorted(bit_of(r) for r in term)) for term in p.affinity_required)
        pref = tuple((int(w), tuple(sorted(bit_of(r) for r in term))) for w, term in p.affinity_preferred)
        tol_h = tuple(sorted(i for k, i in hard_taints.items() if any(t.tolerates(Taint(*k)) for t in p.tolerations)))
        soft_tols = [t for t in p.tolerations if t.effect in ("", "PreferNoSchedule")]
        tol_s = tuple(sorted(i for k, i in soft_taints.items() if any(t.tolerates(Taint(*k)) for t in soft_tols)))
        tol_unsched = any(t.tolerates(Taint("node.kubernetes.io/unschedulable", "", "NoSchedule")) for t in p.tolerations)
        key = (sel, aff, pref, tol_h, tol_s, tol_unsched, bool(p.revocable_zone))
        if key not in class_keys:
            class_keys[key] = len(class_defs)
            class_defs.append(dict(sel=sel, aff=aff, pref=pref, tol_h=tol_h, tol_s=tol_s, unsched=tol_unsched,
                                   revocable=bool(p.revocable_zone)))
        task_class.append(class_keys[key])
    if not class_defs:
        class_defs.append(dict(sel=(), aff=(), pref=(), tol_h=(), tol_s=(), unsched=False, revocable=False))
    Wl = max(1, (len(req_bits) + 63) // 64)
    Wt = max(1, (max(len(hard_taints), len(soft_taints)) + 63) // 64)
    if Wl > abi.VC_MAX_WORDS or Wt > abi.VC_MAX_WORDS:
        raise ValueError("too many distinct label requirements / taints")

    N, T, Q = len(nodes), len(task_pods), len(queues)
    s = Snapshot(N, T, J, Q, len(class_defs), role_off[-1], R, K=len(KDIM_NAMES), Wl=Wl, Wt=Wt, Z=len(zones),
                 pods_dim=pods_dim, B=len(bf_pods))
    s.dim_names = dim_names
    s.node_names = [n.name for n in nodes]
    s.task_keys = [p.key for p in task_pods]
    s.backfill_task_keys = [p.key for p in bf_pods]
    s.job_names = job_ids
    s.queue_names = [q.name for q in queues]

    def setbits(arr_row, bits):
        for b in bits:
            arr_row[b // 64] |= np.uint64(1) << np.uint64(b % 64)

    for c, cd in enumerate(class_defs):
        setbits(s.c_selector[c], cd["sel"])
        if len(cd["aff"]) > abi.VC_MAX_TERMS or len(cd["pref"]) > abi.VC_MAX_TERMS:
            raise ValueError("too many affinity terms")
        s.c_n_affinity[c] = len(cd["aff"])
        for k, term in enumerate(cd["aff"]):
            setbits(s.c_affinity[c, k], term)
        s.c_n_preferred[c] = len(cd["pref"])
        for k, (w, term) in enumerate(cd["pref"]):
            setbits(s.c_preferred[c, k], term)
            s.c_preferred_weight[c, k] = w
        setbits(s.c_tolerated_hard[c], cd["tol_h"])
        setbits(s.c_tolerated_soft[c], cd["tol_s"])
        s.c_flags[c] = (abi.VC_CLASS_REVOCABLE if cd["revocable"] else 0) | \
                       (abi.VC_CLASS_TOLERATES_UNSCHEDULABLE if cd["unsched"] else 0)

    # ---- nodes: NodeInfo.setNodeState / AddTask accounting (api/node_info.go:395-484) -------
    nidx = {n.name: i for i, n in enumerate(nodes)}
    reqs_by_bit = {b: NodeSelectorRequirement(k[0], k[1], k[2]) for k, b in req_bits.items()}
    for i, n in enumerate(nodes):
        v, _ = _resource_vector(n.allocatable, dim_names)
        s.n_allocatable[:, i] = v
        s.n_idle[:, i] = v
        s.n_max_tasks[i] = quantity_value(n.allocatable["pods"]) if "pods" in n.allocatable else 0
        s.n_k8s_allocatable[:, i] = _k8s_vector(n.allocatable, False)
        for b, rq in reqs_by_bit.items():
            if rq.matches(n.labels):
                s.n_label_bits[b // 64, i] |= np.uint64(1) << np.uint64(b % 64)
        for t in n.taints:
            if t.effect == "PreferNoSchedule":
                b = soft_taints[(t.key, t.value, t.effect)]
                s.n_taint_soft[b // 64, i] |= np.uint64(1) << np.uint64(b % 64)
            else:
                b = hard_taints[(t.key, t.value, t.effect)]
                s.n_taint_hard[b // 64, i] |= np.uint64(1) << np.uint64(b % 64)
        if n.unschedulable:
            s.n_flags[i] |= abi.VC_NODE_UNSCHEDULABLE
        if n.revocable_zone:
            s.n_revocable_zone[i] = zones[n.revocable_zone]
    if tdm_zone_active is None:  # derive from the tdm plugin's arguments at "now", as OnSessionOpen does
        tdm_zone_active = {}
        for tier in conf.tiers:
            for po in tier:
                if po.name == "tdm":
                    tdm_zone_active.update(tdm_zones_active(po.arguments))
    for z, zi in zones.items():
        s.zone_active[zi] = 1 if tdm_zone_active.get(z, False) else 0
    for p in pods:
        if not p.node_name or p.node_name not in nidx:
            continue
        st = get_task_status(p)
        if st in ("Succeeded", "Failed"):
            # terminated pods hold no resources: the cache adds a pod to its node unless isTerminated(status)
            # (cache/event_handlers.go:65-67,228-233); a pod in Unknown phase still occupies the node
            continue
        i = nidx[p.node_name]
        v, _ = pod_req(p)
        if st == "Releasing":
            s.n_idle[:, i] -= v
            s.n_releasing[:, i] += v
            s.n_used[:, i] += v
        elif st == "Pipelined":
            s.n_pipelined[:, i] += v
        else:
            s.n_idle[:, i] -= v
            s.n_used[:, i] += v
        s.n_pod_count[i] += 1
        s.n_k8s_requested[:, i] += _k8s_vector(p.requests, False)
        s.n_k8s_nonzero_requested[:, i] += _k8s_vector(p.requests, True)

    # ---- tasks -------------------------------------------------------------------------------
    def fill_tasks(pre, plist, pjob, pclass):
        g = lambda name: getattr(s, pre + name)
        uid_order = np.argsort(np.array([p.uid for p in plist], dtype=object), kind="stable") if plist else []
        for rank, t in enumerate(uid_order):
            g("uid_rank")[t] = rank
        for t, p in enumerate(plist):
            v, has = pod_req(p)
            g("resreq")[:, t] = v
            g("req_has")[t] = has
            g("k8s_req")[:, t] = _k8s_vector(p.requests, False)
            g("k8s_nonzero_req")[:, t] = _k8s_vector(p.requests, True)
            j = pjob[t]
            g("job")[t] = j
            g("klass")[t] = pclass[t]
            g("role")[t] = role_rows[j][get_task_role(p)]
            prio = 1  # api/job_info.go:203,219-227
            if p.priority is not None:
                prio = p.priority
            if TASK_PRIORITY_ANNOTATION in p.annotations:
                try:
                    prio = int(p.annotations[TASK_PRIORITY_ANNOTATION])
                except ValueError:
                    pass
            g("priority")[t] = prio
            g("pod_index")[t] = pod_index_under_task(p.name)
            g("creation_ts")[t] = p.creation_ts

    fill_tasks("t_", task_pods, task_job, task_class[:T])
    fill_tasks("b_", bf_pods, bf_job, task_class[T:])
    for t, p in enumerate(task_pods):
        if p.preemption_policy == "Never":
            s.t_flags[t] |= abi.VC_TASK_PREEMPT_NEVER
        if p.nominated_node_name:  # a node that is not in the session counts as none (allocate.go:627 `ok`)
            s.t_nominated[t] = nidx.get(p.nominated_node_name, -1)
    # node.Tasks: the pods that can become victims (api.PreemptableStatus: Bound | Running, api/helpers.go:70-77)
    run_pods = [p for p in pods if p.node_name in nidx and get_task_status(p) in ("Running", "Bound")]
    s.set_running(len(run_pods))
    uid_order = np.argsort(np.array([p.uid for p in run_pods], dtype=object), kind="stable") if run_pods else []
    for rank, r in enumerate(uid_order):
        s.rt_uid_rank[r] = rank
    for r, p in enumerate(run_pods):
        v, has = pod_req(p)
        s.running_task_keys[r] = p.key
        s.rt_node[r] = nidx[p.node_name]
        j = jidx.get(f"{p.namespace}/{p.group_name}", -1)
        s.rt_job[r] = j
        s.rt_role[r] = role_rows[j][get_task_role(p)] if j >= 0 else -1
        prio = 1
        if p.priority is not None:
            prio = p.priority
        if TASK_PRIORITY_ANNOTATION in p.annotations:
            try:
                prio = int(p.annotations[TASK_PRIORITY_ANNOTATION])
            except ValueError:
                pass
        s.rt_priority[r] = prio
        s.rt_pod_index[r] = pod_index_under_task(p.name)
        s.rt_creation_ts[r] = p.creation_ts
        s.rt_resreq[:, r] = v
        s.rt_req_has[r] = has
        s.rt_k8s_req[:, r] = _k8s_vector(p.requests, False)
        s.rt_k8s_nonzero_req[:, r] = _k8s_vector(p.requests, True)
        fl = abi.VC_RT_RUNNING if get_task_status(p) == "Running" else abi.VC_RT_BOUND
        if pod_preemptable(p):
            fl |= abi.VC_RT_PREEMPTABLE
        if is_best_effort(v):
            fl |= abi.VC_RT_BEST_EFFORT
        if pod_critical(p):
            fl |= abi.VC_RT_CRITICAL
        s.rt_flags[r] = fl

    # ---- jobs --------------------------------------------------------------------------------
    uid_order = sorted(range(J), key=lambda j: job_ids[j])
    for rank, j in enumerate(uid_order):
        s.j_uid_rank[j] = rank
    for j, pg in enumerate(podgroups):
        s.j_queue[j] = qidx.get(pg.queue, -1)
        s.j_min_available[j] = pg.min_member
        s.j_priority[j] = pg.priority
        s.j_creation_ts[j] = pg.creation_ts
        fl = 0
        if pg.phase in ("Pending", ""):
            fl |= abi.VC_JOB_PENDING_PHASE
        if pg.preemptable:
            fl |= abi.VC_JOB_PREEMPTABLE
        if pg.unsupported:
            fl |= abi.VC_JOB_UNSUPPORTED
        s.j_flags[j] = fl
    s.j_n_tasks_total[:] = snap_j["ntasks"]
    s.j_ready_num[:] = snap_j["ready"]
    s.j_waiting_num[:] = snap_j["waiting"]
    s.j_pending_besteffort[:] = snap_j["pbe"]
    s.j_valid_num[:] = snap_j["valid"]
    s.j_task_min_total[:] = snap_j["tmt"]
    s.j_role_off[:] = np.array(role_off, np.int32)
    s.j_allocated[:] = j_alloc
    s.r_min[:] = role_tables["min"]
    s.r_occupied[:] = role_tables["occ"]
    s.r_pipelined[:] = role_tables["pip"]
    s.r_pending_other[:] = role_tables["pending_other"]
    s.r_valid[:] = role_tables["valid"]
    s.r_flags[:] = role_tables["flags"]

    # ---- queues: proportion's allocated / request sums (proportion.go:143-156) --------------
    uid_order = sorted(range(Q), key=lambda q: queues[q].name)
    for rank, q in enumerate(uid_order):
        s.q_uid_rank[q] = rank
    for qi, q in enumerate(queues):
        s.q_weight[qi] = q.weight
        s.q_priority[qi] = q.priority
        s.q_creation_ts[qi] = q.creation_ts
        s.q_flags[qi] = (abi.VC_QUEUE_OPEN if q.state == "Open" else 0) | (0 if q.reclaimable else abi.VC_QUEUE_NOT_RECLAIMABLE)
        if q.capability:
            v, has = _resource_vector(q.capability, dim_names)
            s.q_capability[:, qi] = v
            s.q_capability_has[qi] = has | abi.VC_RES_HAS_ANY
        if q.guarantee:
            v, has = _resource_vector(q.guarantee, dim_names)
            s.q_guarantee[:, qi] = v
            s.q_guarantee_has[qi] = has | abi.VC_RES_HAS_ANY
    for j, pg in enumerate(podgroups):
        qi = qidx.get(pg.queue, -1)
        if qi < 0:
            continue
        for p in job_pods[j]:
            st = get_task_status(p)
            v, has = pod_req(p)
            if allocated_status(st):
                s.q_allocated[:, qi] += v
                s.q_allocated_has[qi] |= has
                s.q_request[:, qi] += v
                s.q_request_has[qi] |= has
            elif st == "Pending":
                s.q_request[:, qi] += v
                s.q_request_has[qi] |= has
    s.conf = build_conf(conf, dim_names, KDIM_NAMES)
    s.actions = tuple(conf.actions)
    if hypernodes is not None:
        encode_hypernodes(s, hypernodes, podgroups, job_pods)
    return s
