"""Node-level view of a GPU federation, and launch helpers.

In the reference a *node* is a server process with a private dataset; a model that pools N nodes
creates N clients/Ops and lets the graph add the log-potentials
(``/root/reference/demo_model.py:17-36``, README "distributed" diagram).  Here the N nodes are the
N data shards resident on the GPUs of one NVSwitch domain, and :class:`NodeFederation` gives each
of them the reference's call signatures:

* ``fed.evaluate_node(i, intercept, slope) -> (logp, [grads])`` — one node's ``LogpGradFunc``;
* ``fed.evaluate_nodes({i: inputs, ...})`` — several nodes in ONE fused launch (what a fused
  ``ParallelAsyncOp`` of :class:`~pytensor_federated_b200.wrapper_ops.FederatedLogpGradOp`
  children calls);
* ``fed.node_ops()`` — one ``FederatedLogpGradOp`` per node for building models;
* ``fed.register_services("gpu")`` — makes ``LogpGradServiceClient("gpu", i)`` resolve to node i
  without sockets (the reference's client API, the NVLink data plane).
"""
from __future__ import annotations

import contextlib
import os
import socket
import threading
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np

from .models.linreg import LinregShards
from .parallel.engine import FederatedEngine, FederationError


class NodeFederation:
    """Per-node access to an engine whose model keeps per-node results.

    * ``LinregShards`` — node = shard; inputs ``(intercept, slope)``.
    * ``OdeShards(..., node_ids=, n_nodes=)`` — node = the shards with that node id; input ``(theta,)``; every
      node may be given its own parameter vector.
    * ``GlmShards(..., node_ids=, n_nodes=)`` — node = the segments with that node id; inputs
      ``(intercepts[G], beta[P])`` — plus ``phi[D]`` for the families with fitted parameters (negative binomial,
      Student-t, normal).  Nodes that are given the same parameters (the usual federated GLM)
      share a chain; *distinct* parameter vectors occupy one chain each, so the model must have been built
      with ``n_chains >=`` the number of distinct vectors of a call.

    Whatever the model, one call of :meth:`evaluate_nodes` is ONE fused launch per GPU.
    """

    def __init__(self, engine: FederatedEngine) -> None:
        from .models.glm import GlmShards
        from .models.ode import OdeShards

        m = engine.model
        if isinstance(m, LinregShards):
            self._kind = "linreg"
            self.n_nodes = m.n_shards_total
            self._intercepts = np.zeros(self.n_nodes)
            self._slopes = np.zeros(self.n_nodes)
        elif isinstance(m, OdeShards) and m.node_ids is not None:
            self._kind = "ode"
            self.n_nodes = m.n_nodes
            self._theta = np.zeros((m.n_nodes, m.n_params))
        elif isinstance(m, GlmShards) and m.node_ids is not None:
            self._kind = "glm"
            self.n_nodes = m.n_nodes
        else:
            raise FederationError(
                "NodeFederation needs a model that keeps per-node results: LinregShards, or OdeShards / GlmShards "
                "built with node_ids= and n_nodes="
            )
        self.engine = engine
        self._lock = threading.Lock()   # parameter staging + launch + un-staging of the result form one unit
        self.n_launches = 0

    # -- evaluation ----------------------------------------------------------------------------
    def evaluate_nodes(self, requests: Dict[int, Sequence[np.ndarray]]) -> Dict[int, Tuple[np.ndarray, List[np.ndarray]]]:
        """``{node: inputs} -> {node: (logp, [gradients])}``, one launch."""
        for node in requests:
            if not 0 <= int(node) < self.n_nodes:
                raise FederationError(f"node {node} does not exist (the federation has {self.n_nodes})")
        with self._lock:
            self.n_launches += 1
            return getattr(self, f"_evaluate_{self._kind}")(requests)

    def _evaluate_linreg(self, requests):
        for node, (a, b) in requests.items():
            self._intercepts[node] = a.item() if hasattr(a, "item") else float(np.asarray(a))
            self._slopes[node] = b.item() if hasattr(b, "item") else float(np.asarray(b))
        per = LinregShards.per_shard(self.engine.evaluate_raw([self._intercepts, self._slopes]))
        return {node: (np.array(per[node, 0]), [np.array(per[node, 1]), np.array(per[node, 2])]) for node in requests}

    def _evaluate_ode(self, requests):
        m = self.engine.model
        for node, inputs in requests.items():
            (theta,) = inputs
            self._theta[node] = np.asarray(theta, dtype=np.float64).reshape(m.n_params)
        per = m.per_node(self.engine.evaluate_raw([self._theta]))
        return {node: (np.array(per[node, 0]), [per[node, 1:].copy()]) for node in requests}

    def _evaluate_glm(self, requests):
        m = self.engine.model
        G, K, D = m.n_groups, m.n_chains, m.n_family_params
        GP = G + m.n_features
        chains: Dict[bytes, int] = {}      # distinct parameter vector [intercept, beta, phi] -> chain
        rows: List[np.ndarray] = []
        chain_of: Dict[int, int] = {}
        shapes: Dict[int, tuple] = {}
        phi_shapes: Dict[int, tuple] = {}
        for node, inputs in requests.items():
            if len(inputs) != m.n_inputs:
                raise ValueError(f"node {node}: the {m.family} GLM takes {m.n_inputs} inputs, got {len(inputs)}")
            ic = np.asarray(inputs[0], dtype=np.float32)
            parts = [ic.reshape(G), np.asarray(inputs[1], dtype=np.float32).reshape(m.n_features)]
            if D:
                parts.append(np.asarray(inputs[2], dtype=np.float32).reshape(D))
                phi_shapes[node] = np.shape(inputs[2])   # a scalar phi (D = 1) gets a scalar gradient
            vec = np.concatenate(parts)
            key = vec.tobytes()
            if key not in chains:
                if len(rows) == K:
                    raise FederationError(
                        f"{len(rows) + 1} distinct parameter vectors in one call but the model evaluates {K} chain(s) per "
                        "launch: build GlmShards with n_chains >= the number of nodes that get their own parameters"
                    )
                chains[key] = len(rows)
                rows.append(vec)
            chain_of[node] = chains[key]
            shapes[node] = ic.shape
        theta = np.stack(rows + [rows[0]] * (K - len(rows)))                       # unused chains repeat the first
        th = theta if K > 1 else theta[0]
        inputs = [th[..., :G], th[..., G:GP]] + ([th[..., GP:]] if D else [])
        per = m.per_node(self.engine.evaluate_raw(inputs))                         # [n_nodes, K, 1 + G + P + D]
        out = {}
        for node in requests:
            v = per[node, chain_of[node]]
            grads = [v[1 : 1 + G].reshape(shapes[node]).copy(), v[1 + G : 1 + GP].copy()]
            out[node] = (np.array(v[0]), grads + ([v[1 + GP :].reshape(phi_shapes[node]).copy()] if D else []))
        return out

    def evaluate_node(self, node: int, *inputs) -> Tuple[np.ndarray, List[np.ndarray]]:
        return self.evaluate_nodes({node: inputs})[node]

    def logp_grad_func(self, node: int) -> Callable:
        """The node as a plain ``LogpGradFunc`` (usable with the generic ``LogpGradOp``)."""
        return lambda *inputs: self.evaluate_node(node, *inputs)

    def compute_func(self, node: int) -> Callable:
        """The node as a ``ComputeFunc``: ``(logp, *gradients)``."""

        def compute(*inputs):
            logp, grads = self.evaluate_node(node, *inputs)
            return (logp, *grads)

        return compute

    def all_nodes_func(self) -> Callable:
        """The WHOLE federation as one ``LogpGradFunc`` — node parameters stacked along a leading axis, the
        summed log-likelihood and per-node gradients back, one launch:

        * linear regression: ``f(intercepts, slopes) -> (logp, [d_intercepts, d_slopes])``, each argument a vector
          ``[n_nodes]`` or a scalar shared by all nodes (its gradient is then the sum over the nodes);
        * ODE: ``f(theta[n_nodes, n_params]) -> (logp, [d_theta])``;
        * GLM (parameters shared by the nodes): ``f(intercept, beta) -> (logp, [d_intercept, d_beta])``, and for the
          families with fitted parameters ``f(intercept, beta, phi) -> (logp, [d_intercept, d_beta, d_phi])``.

        With :meth:`all_nodes_op` the model graph has ONE federated node instead of one per data holder, so the
        Python cost of a model evaluation no longer grows with the size of the federation."""
        kind, eng = self._kind, self.engine
        if kind == "linreg":
            def func(intercepts, slopes):
                # a scalar argument is shared by all nodes and gets the summed gradient (LinregShards.unpack_result)
                with self._lock:
                    self.n_launches += 1
                    logp, da, db = eng.evaluate(intercepts, slopes)
                    return logp, [da, db]
        elif kind == "ode":
            def func(theta):
                m = eng.model
                with self._lock:
                    self.n_launches += 1
                    th = np.broadcast_to(np.asarray(theta, dtype=np.float64), (self.n_nodes, m.n_params))
                    per = m.per_node(eng.evaluate_raw([th]))
                    return np.asarray(per[:, 0].sum()), [per[:, 1:].copy()]
        elif eng.model.n_family_params:
            def func(intercept, beta, phi):
                with self._lock:
                    self.n_launches += 1
                    logp, *grads = eng.evaluate(intercept, beta, phi)
                    return logp, grads
        else:
            def func(intercept, beta):
                with self._lock:
                    self.n_launches += 1
                    logp, *grads = eng.evaluate(intercept, beta)
                    return logp, grads
        return func

    # -- graph integration ---------------------------------------------------------------------
    def node_ops(self):
        from .wrapper_ops import FederatedLogpGradOp

        return [FederatedLogpGradOp(self, i) for i in range(self.n_nodes)]

    def all_nodes_op(self):
        """One ``LogpGradOp`` over :meth:`all_nodes_func` (vector parameters in, summed logp and vector gradients out)."""
        from .wrapper_ops import LogpGradOp

        return LogpGradOp(self.all_nodes_func())

    # -- reference client API ------------------------------------------------------------------
    def register_services(self, host: str = "gpu", first_port: int = 0) -> List[Tuple[str, int]]:
        from . import service

        addresses = []
        for i in range(self.n_nodes):
            service.register_local_node(host, first_port + i, self.compute_func(i), name=f"{host}:{first_port + i}")
            addresses.append((host, first_port + i))
        self._registered = addresses
        return addresses

    def unregister_services(self) -> None:
        from . import service

        for host, port in getattr(self, "_registered", []):
            service.unregister_local_node(host, port)
        self._registered = []

    def shutdown(self) -> None:
        self.unregister_services()
        self.engine.shutdown()


def register_replicas(engines: Sequence[FederatedEngine], host: str = "gpu", first_port: int = 0) -> List[Tuple[str, int]]:
    """Replicated-shard mode: every engine holds a REPLICA of the same data (typically one per GPU); they are
    registered as in-process nodes ``(host, first_port + i)`` and the returned address list goes to
    ``ArraysToArraysServiceClient(hosts_and_ports=...)`` / ``LogpGradServiceClient(hosts_and_ports=...)``.

    The client then behaves as it does towards replicated gRPC servers in the reference
    (``/root/reference/pytensor_federated/service.py:239-275``, ``:407-416``): it connects to the replica with
    the fewest clients (chains of a sampler spread over the GPUs), and when a replica is lost — its engine shut
    down or timed out — the call is retried on a surviving one.  A *sharded* federation cannot do that (a lost
    shard is lost data); replicas trade HBM for availability and for chain-level parallelism."""
    from . import service

    addresses = []
    for i, eng in enumerate(engines):
        service.register_local_node(host, first_port + i, eng.evaluate, name=f"{host}:{first_port + i}")
        addresses.append((host, first_port + i))
    return addresses


def free_port() -> int:
    """An unused TCP port on 127.0.0.1 (rendezvous of a freshly launched federation)."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _peer_main(rank: int, world: int, port: int, build_model, backend: str, device_type: str, timeout: float) -> None:
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    if device_type == "cuda":
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dev = torch.device("cpu")
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        model = build_model(rank, world, dev)
        eng = FederatedEngine(model, backend=backend, device=dev, timeout=timeout)
        eng.serve()
        eng.shutdown()
    finally:
        dist.destroy_process_group()


@contextlib.contextmanager
def launch_federation(build_model: Callable, n_nodes: int, *, device_type: Optional[str] = None,
                      backend: str = "auto", timeout: float = 3600.0, speculative_us: Optional[float] = None):
    """Starts ``n_nodes - 1`` peer processes (one per GPU) and yields the root's engine.

    ``build_model(rank, world, device) -> ShardModel`` builds each node's private shard model and
    must be picklable (module-level function).  The calling process is rank 0, the client.  On
    exit the peers are drained and joined.  ``device_type="cpu"`` runs the same topology over
    gloo with the collective backend (plumbing tests).  ``speculative_us`` > 0 lets the root keep the next
    evaluation's kernel enqueued ahead of theta (:meth:`FederatedEngine.set_speculative`; fused backend only).
    """
    import torch
    import torch.distributed as dist
    import torch.multiprocessing as mp

    if device_type is None:
        device_type = "cuda" if torch.cuda.is_available() else "cpu"
    if device_type == "cuda" and torch.cuda.device_count() < n_nodes:
        raise FederationError(f"{n_nodes} nodes requested but only {torch.cuda.device_count()} GPUs are visible")
    port = free_port()
    ctx = mp.get_context("spawn")
    procs = [
        ctx.Process(target=_peer_main, args=(r, n_nodes, port, build_model, backend, device_type, timeout), daemon=True)
        for r in range(1, n_nodes)
    ]
    for p in procs:
        p.start()
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    owns_pg = False
    engine = None
    try:
        if n_nodes > 1:
            if device_type == "cuda":
                torch.cuda.set_device(0)
                dist.init_process_group("nccl", rank=0, world_size=n_nodes, device_id=torch.device("cuda", 0))
            else:
                dist.init_process_group("gloo", rank=0, world_size=n_nodes)
            owns_pg = True
        dev = torch.device("cuda", 0) if device_type == "cuda" else torch.device("cpu")
        engine = FederatedEngine(build_model(0, n_nodes, dev), backend=backend, device=dev, timeout=timeout,
                                 speculative_us=speculative_us)
        yield engine
    finally:
        if engine is not None:
            engine.shutdown()
        if owns_pg:
            dist.destroy_process_group()
        for p in procs:
            p.join(60)
            if p.is_alive():
                p.terminate()


__all__ = ["NodeFederation", "launch_federation", "register_replicas", "free_port"]
