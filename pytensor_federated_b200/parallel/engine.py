"""Federation engine: ``theta -> [LL, dLL/dtheta]`` over all nodes of an NVSwitch domain.

Two interchangeable data planes behind one interface:

``backend="fused"`` (the product)
    One hand-written sm_100a kernel per GPU does broadcast -> compute -> reduce with in-kernel
    NVLink stores/multicast (``csrc/fed_comm.cuh``).  The root's host thread only memcpy's theta
    into pinned memory, launches, and spins on a pinned completion flag; peer hosts pre-enqueue
    kernels that wait on the device.  No NCCL call, no serialisation, no RPC on the path.

``backend="collective"`` (the baseline, also the CPU/gloo plumbing path)
    ``dist.broadcast(theta)`` -> eager PyTorch compute of the node partial ->
    ``dist.reduce(partials)``.  This is what BASELINE.json calls "the baseline, not the product";
    it doubles as the oracle in multi-process tests and runs on CPU with gloo.

The reference's equivalent of one ``evaluate`` call is N concurrent gRPC round trips plus a
client-side sum (``/root/reference/pytensor_federated/op_async.py:114-130``,
``service.py:150-158``).
"""
from __future__ import annotations

import ctypes as C
import logging
import os
import threading
from typing import List, Optional, Sequence, Tuple

import numpy as np

from ..models.base import ShardModel

_log = logging.getLogger(__name__)

_STOP = -1.0


class FederationError(RuntimeError):
    """The engine was misused or the native runtime reported a failure (message carries the native error)."""


class EngineClosedError(FederationError):
    """The engine was shut down.  A client that reaches it through the local node registry treats this like a
    lost connection and fails over to another replica."""

    marks_node_lost = True


class FederationTimeout(TimeoutError):
    """A node did not answer within the engine timeout (dead peer / lost shard)."""

    marks_node_lost = True


def _dist():
    import torch.distributed as dist

    return dist


class FederatedEngine:
    """Evaluates a :class:`ShardModel` across the ranks of a process group.

    Rank 0 is the *root* (the client's GPU): it calls :meth:`evaluate`.  Every other rank calls
    :meth:`serve`, which returns when the root calls :meth:`shutdown`.
    With ``group=None`` and no initialised ``torch.distributed`` the engine is single-node.
    """

    def __init__(
        self,
        model: ShardModel,
        *,
        backend: str = "auto",
        group=None,
        device=None,
        timeout: Optional[float] = None,
        idle_timeout: Optional[float] = None,
        comm: Optional[str] = None,
        grid: Optional[int] = None,
        speculative_us: Optional[float] = None,
    ) -> None:
        import torch

        from ..config import get_config

        cfg = get_config()
        timeout = cfg.timeout if timeout is None else timeout
        # ``timeout`` bounds ONE evaluation (a dead peer / lost theta inside an evaluation in flight).  A client
        # that merely pauses between evaluations is not a failure: peers re-arm their waiting kernels for as long
        # as ``idle_timeout`` allows (0 = for ever; B200FED_IDLE_TIMEOUT)
        self.idle_timeout = float(cfg.idle_timeout if idle_timeout is None else idle_timeout)
        self._serve_ahead = cfg.serve_ahead
        self._speculative_us = float(cfg.speculative_us if speculative_us is None else speculative_us)
        #: True while the root keeps kernels enqueued ahead of the next theta (see :meth:`set_speculative`)
        self.speculative = False

        self.model = model
        dist = _dist()
        self._dist_ready = dist.is_available() and dist.is_initialized()
        self.group = group
        self.rank = dist.get_rank(group) if self._dist_ready else 0
        self.world = dist.get_world_size(group) if self._dist_ready else 1
        if device is None:
            device = getattr(model, "device", None) or torch.device("cpu")
        self.device = torch.device(device)
        if backend == "auto":
            backend = "fused" if self.device.type == "cuda" else "collective"
        if backend not in ("fused", "collective"):
            raise ValueError(f"unknown backend {backend!r}")
        if backend == "fused" and self.device.type != "cuda":
            raise FederationError("the fused backend needs a CUDA device; use backend='collective' on CPU")
        self.backend = backend
        self.timeout = float(timeout)
        self._lock = threading.Lock()
        self._closed = False
        self._handle = None
        self._keepalive = []
        self._ipc_opened: List[int] = []  # peer blocks mapped with cudaIpcOpenMemHandle (closed in shutdown)
        self.comm_mode = "none"
        self.n_evals = 0
        self._stop_seen = False
        # host-side tracing: NVTX range per evaluation (B200FED_NVTX=1); device-side phase stamps: trace()
        self._nvtx = bool(os.environ.get("B200FED_NVTX")) and self.device.type == "cuda"
        if backend == "fused":
            self._init_fused(comm or cfg.comm, grid)

    # ------------------------------------------------------------------ fused backend
    def _init_fused(self, comm: str, grid: Optional[int]) -> None:
        import torch

        from ..ops import native

        lib = native.load()
        self._lib = lib
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        m = self.model
        handle = lib.b200_engine_create(dev_index, self.rank, self.world, m.n_theta_words, m.n_vals, 0)
        if not handle:
            raise FederationError(f"engine creation failed: {native.last_error()}")
        self._handle = C.c_void_p(handle)
        self._dev_index = dev_index
        torch.cuda.synchronize(self.device)  # model tensors were produced on torch's streams
        m.attach(lib, self._handle)
        if grid:
            lib.b200_engine_set_grid(self._handle, int(grid))
        lib.b200_engine_set_timeout(self._handle, self.timeout)
        lib.b200_engine_set_idle_timeout(self._handle, self.idle_timeout)
        self._bootstrap_comm(comm)
        native.check(lib.b200_engine_reset(self._handle), "engine reset")
        if self.world > 1:
            _dist().barrier(group=self.group)
        # staging buffers handed to the native eval call (which copies into / out of pinned memory)
        self._stage = np.zeros(max(1, m.n_theta_words), dtype=np.uint32)
        self._out = np.zeros(m.n_vals, dtype=np.float64)
        self._stage_p = self._stage.ctypes.data_as(C.c_void_p)
        self._out_p = self._out.ctypes.data_as(C.c_void_p)
        if self._speculative_us > 0 and self.rank == 0:
            self.set_speculative(self._speculative_us)

    def set_speculative(self, wait_us: float = 1000.0) -> bool:
        """Root, fused backend: keep the NEXT evaluation's kernel enqueued while the client is still thinking.

        ``evaluate`` then finds a kernel that is already resident, set up, with its first tiles loaded and
        polling host memory for theta (tagged words over PCIe), and enqueues the one after it while the GPU
        computes — launch latency, kernel start-up and the first loads leave the sequential path of a sampler
        (~7 us per evaluation).  A kernel whose theta does not arrive within ``wait_us`` gives up (an idle tick,
        exactly like a peer between sampling phases) and the next ``evaluate`` launches afresh, so the GPU spins
        for at most ``2 x wait_us`` after the last evaluation; other work queued on this GPU waits that long.
        ``wait_us=0`` switches back to one launch per evaluation.  Needs theta as tagged words (at most 1024
        32-bit words); returns whether speculation is on.
        """
        from ..ops import native

        if self.backend != "fused" or not self.is_root:
            return False
        with self._lock:
            rc = int(self._lib.b200_engine_set_speculative(self._handle, float(wait_us)))
            if rc < 0:
                raise FederationError(f"set_speculative failed (rc={rc}): {native.last_error()}")
            self.speculative = rc == 1
            return self.speculative

    def _bootstrap_comm(self, comm: str) -> None:
        """Makes every node's comm block addressable from this process.

        ``symm``: torch symmetric memory (CUDA VMM; also yields the NVSwitch multicast alias used
        by ``multimem.st``).  ``ipc``: cudaMalloc + CUDA IPC handles exchanged over the process
        group.  ``auto`` tries ``symm`` and falls back to ``ipc``.
        """
        import torch

        from ..ops import native

        lib = self._lib
        m = self.model
        if self.world == 1:
            ptr = C.c_void_p()
            native.check(lib.b200_engine_alloc_comm(self._handle, C.byref(ptr)), "alloc comm")
            peers = native.void_p_array([ptr.value])
            native.check(lib.b200_engine_bind_comm(self._handle, ptr, peers, None), "bind comm")
            self.comm_mode = "local"
            return
        dist = _dist()
        nbytes = int(lib.b200_comm_block_bytes(self.world, m.n_theta_words, m.n_vals))
        if comm in ("auto", "symm"):
            try:
                import torch.distributed._symmetric_memory as symm_mem

                buf = symm_mem.empty(nbytes, dtype=torch.uint8, device=self.device)
                buf.zero_()
                torch.cuda.synchronize(self.device)
                pg = self.group if self.group is not None else dist.group.WORLD
                hdl = symm_mem.rendezvous(buf, pg.group_name)
                ptrs = [int(p) for p in hdl.buffer_ptrs]
                mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
                if os.environ.get("B200FED_NO_MULTICAST"):
                    mc = 0
                native.check(
                    lib.b200_engine_bind_comm(
                        self._handle, C.c_void_p(buf.data_ptr()), native.void_p_array(ptrs),
                        C.c_void_p(mc) if mc else None,
                    ),
                    "bind comm",
                )
                self._keepalive += [buf, hdl]
                self.comm_mode = "symm+multicast" if mc else "symm"
                ok = 1
            except Exception as ex:  # noqa: BLE001 - any failure means "try IPC"
                if comm == "symm":
                    raise
                _log.warning("symmetric-memory bootstrap failed (%s); falling back to CUDA IPC", ex)
                ok = 0
            flag = torch.tensor([ok], device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
            if int(flag.item()) == 1:
                return
        # CUDA IPC
        ptr = C.c_void_p()
        native.check(lib.b200_engine_alloc_comm(self._handle, C.byref(ptr)), "alloc comm")
        hbuf = C.create_string_buffer(64)
        native.check(lib.b200_ipc_get_handle(ptr, hbuf), "ipc get handle")
        handles: List[Optional[bytes]] = [None] * self.world
        dist.all_gather_object(handles, hbuf.raw, group=self.group)
        ptrs = []
        for r, hb in enumerate(handles):
            if r == self.rank:
                ptrs.append(ptr.value)
                continue
            out = C.c_void_p()
            native.check(lib.b200_ipc_open_handle(self._dev_index, hb, C.byref(out)), f"ipc open rank {r}")
            ptrs.append(out.value)
            self._ipc_opened.append(out.value)
        native.check(lib.b200_engine_bind_comm(self._handle, ptr, native.void_p_array(ptrs), None), "bind comm")
        self.comm_mode = "ipc"

    # ------------------------------------------------------------------ evaluation
    @property
    def is_root(self) -> bool:
        return self.rank == 0

    def _evaluate_locked(self, inputs: Sequence[np.ndarray]):
        """One evaluation with ``self._lock`` held by the caller: returns ``(vals, ctx)`` where ``vals``
        is the engine's shared ``float64[n_vals]`` buffer (valid until the lock is released) and
        ``ctx`` the model's per-call context for ``unpack_result``."""
        if self._closed:
            raise EngineClosedError("engine is shut down")
        if not self.is_root:
            raise FederationError("only rank 0 evaluates; other ranks call serve()")
        self.n_evals += 1
        if self._nvtx:
            import torch

            torch.cuda.nvtx.range_push(f"fed_eval[{self.n_evals}]")
        try:
            if self.backend == "fused":
                ctx = self.model.pack_theta(inputs, self._stage)
                rc = self._lib.b200_engine_eval(
                    self._handle, self._stage_p, self.model.n_theta_words, self._out_p, self.timeout + 5.0
                )
                if rc != 0:
                    self._raise(rc)
                return self._out, ctx
            return self._collective_eval(inputs), self.model.call_context(inputs)
        finally:
            if self._nvtx:
                torch.cuda.nvtx.range_pop()

    def evaluate_raw(self, inputs: Sequence[np.ndarray]) -> np.ndarray:
        """Root: one federated evaluation, returns a fresh copy of the reduced ``float64[n_vals]``."""
        with self._lock:
            vals, _ = self._evaluate_locked(inputs)
            return np.array(vals, dtype=np.float64, copy=True)

    def evaluate(self, *inputs: np.ndarray) -> List[np.ndarray]:
        """``ComputeFunc`` signature: ``(logp, *gradients)`` as fresh NumPy arrays.

        Thread-safe: packing, the launch and the unpacking of the shared result buffer happen
        under one lock, and the shapes of THIS call's inputs travel with the call (several service
        streams or a ``DynamicBatcher`` may call this concurrently)."""
        with self._lock:
            vals, ctx = self._evaluate_locked(inputs)
            return self.model.unpack_result(vals, ctx)

    __call__ = evaluate

    def logp_grad(self, *inputs: np.ndarray) -> Tuple[np.ndarray, List[np.ndarray]]:
        logp, *grads = self.evaluate(*inputs)
        return logp, grads

    def _raise(self, rc: int) -> None:
        from ..ops import native

        if rc > 0 and rc & 4:
            raise FederationError(
                "a tensor-core kernel's mbarrier pipeline stalled (internal error; the CUDA context is intact, "
                "the evaluation's result is invalid)"
            )
        if rc > 0:
            which = []
            if rc & 1:
                which.append("theta broadcast never arrived")
            if rc & 2:
                which.append("a peer node did not deliver its partial")
            raise FederationTimeout(
                f"federated evaluation timed out after {self.timeout}s ({'; '.join(which)}). "
                "A lost data shard cannot be failed over."
            )
        if rc == -5:
            raise FederationTimeout(native.last_error())
        raise FederationError(f"native evaluation failed (rc={rc}): {native.last_error()}")

    # device-timed benchmarking hooks (root, fused)
    def launch(self) -> int:
        """Enqueues one evaluation with the current theta (``set_device_theta`` or the last ``evaluate``)
        and returns its epoch without waiting.  Results live in ONE host-mapped buffer: with several
        epochs in flight ``wait`` returns the newest completed result, and models small enough for the
        flag-in-data protocol (``n_vals <= 128``) must ``wait`` for each epoch before launching the next —
        their result words are tagged with the exact epoch."""
        rc = self._lib.b200_engine_launch(self._handle)
        if rc != 0:
            self._raise(rc)
        return int(self._lib.b200_engine_epoch(self._handle))

    def wait(self, epoch: int) -> np.ndarray:
        """Spins on the host-mapped completion flag (or tagged result words) of ``epoch``; see :meth:`launch`."""
        rc = self._lib.b200_engine_wait(self._handle, epoch, self._out_p, self.timeout + 5.0)
        if rc != 0:
            self._raise(rc)
        return self._out

    def set_device_theta(self, inputs: Sequence[np.ndarray], enable: bool = True) -> None:
        """Parks theta in device memory so back-to-back launches need no host traffic."""
        from ..ops import native

        self.model.pack_theta(inputs, self._stage)
        native.check(
            self._lib.b200_engine_set_device_theta(
                self._handle, self._stage_p, self.model.n_theta_words, int(enable)
            ),
            "set_device_theta",
        )

    def torch_stream(self):
        import torch

        return torch.cuda.ExternalStream(int(self._lib.b200_engine_stream(self._handle)), device=self.device)

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.b200_engine_launches(self._handle)) if self._handle else 0

    def trace(self, epoch: int) -> Tuple[int, int, int]:
        buf = (C.c_ulonglong * 4)()
        self._lib.b200_engine_trace(self._handle, epoch, buf)
        return int(buf[0]), int(buf[1]), int(buf[2])

    def enable_cta_trace(self, on: bool = True) -> None:
        """Per-CTA phase stamps (``fed::stamp`` in the kernels) for the following launches."""
        self._lib.b200_engine_enable_cta_trace(self._handle, int(on))

    def cta_trace(self) -> np.ndarray:
        """``uint64[grid, 8]`` device-timer stamps (ns) of the most recent launch on this rank:
        0 entry, 1 theta acquired, 2 setup done, 3 first tile landed, 4 last load issued, 5 main loop
        done, 6 partial stored, 7 exit.  Zero where a kernel has no such phase."""
        rows = int(self._lib.b200_engine_max_blocks(self._handle))
        buf = np.zeros((rows, 8), dtype=np.uint64)
        n = int(self._lib.b200_engine_cta_trace(self._handle, buf.ctypes.data_as(C.POINTER(C.c_ulonglong)), rows))
        if n < 0:
            raise FederationError("cta_trace failed")
        return buf[:n].copy()

    # ------------------------------------------------------------------ collective backend
    def _collective_eval(self, inputs) -> np.ndarray:
        import torch

        m = self.model
        words = np.zeros(max(1, m.n_theta_words), dtype=np.uint32)
        m.pack_theta(inputs, words)
        header = torch.zeros(1 + words.size, dtype=torch.float64)
        header[0] = 1.0
        header[1:] = torch.from_numpy(words.astype(np.float64))
        return self._collective_round(header)

    def _collective_round(self, header) -> Optional[np.ndarray]:
        import torch

        dist = _dist()
        m = self.model
        header = header.to(self.device)
        if self.world > 1:
            dist.broadcast(header, src=dist.get_global_rank(self.group, 0) if self.group else 0, group=self.group)
        if float(header[0]) == _STOP:
            return None
        words = header[1:].cpu().numpy().astype(np.uint32)
        inputs = self._unpack_words(words)
        compute = getattr(m, "eager_partial", None) if self.device.type == "cuda" else None
        compute = compute or m.reference_partial
        partial = torch.from_numpy(np.asarray(compute(inputs), dtype=np.float64)).to(self.device)
        if self.world > 1:
            dist.reduce(partial, dst=dist.get_global_rank(self.group, 0) if self.group else 0, group=self.group)
        return partial.cpu().numpy()

    def _unpack_words(self, words: np.ndarray):
        """Inverse of ``pack_theta`` for peers of the collective path: models expose
        ``inputs_from_words`` when their inputs are not simply the float32 words."""
        fn = getattr(self.model, "inputs_from_words", None)
        if fn is not None:
            return fn(words)
        return default_inputs_from_words(self.model, words)

    # ------------------------------------------------------------------ peers
    def serve(self, max_epochs: int = 0, ahead: Optional[int] = None) -> int:
        """Peer ranks: answer the root's evaluations until it shuts the federation down.

        Returns the number of evaluations served.
        """
        if self.is_root:
            raise FederationError("rank 0 is the client; it does not serve")
        if self.backend == "fused":
            from ..ops import native

            ahead = self._serve_ahead if ahead is None else ahead
            n = int(self._lib.b200_engine_serve(self._handle, int(ahead), int(max_epochs)))
            if n < 0:
                if n == -7:
                    raise FederationTimeout(native.last_error())
                raise FederationError(f"serve loop failed (rc={n}): {native.last_error()}")
            return n
        import torch

        served = 0
        m = self.model
        while max_epochs <= 0 or served < max_epochs:
            header = torch.zeros(1 + max(1, m.n_theta_words), dtype=torch.float64)
            if self._collective_round(header) is None:
                self._stop_seen = True  # the root's shutdown broadcast has been consumed
                break
            served += 1
        return served

    def shutdown(self) -> None:
        """Root: drain the peers.  Everyone: release native resources."""
        if self._closed:
            return
        self._closed = True
        try:
            if self.is_root and self.world > 1:
                if self.backend == "fused":
                    self._lib.b200_engine_stop_peers(self._handle)
                else:
                    import torch

                    header = torch.zeros(1 + max(1, self.model.n_theta_words), dtype=torch.float64)
                    header[0] = _STOP
                    self._collective_round(header)
            elif (not self.is_root) and self.world > 1 and self.backend == "collective" and not self._stop_seen:
                # Collectives must match on every rank: a peer that is not inside serve() (it served a
                # bounded number of epochs) still has to take part in the root's STOP broadcast.
                import torch

                header = torch.zeros(1 + max(1, self.model.n_theta_words), dtype=torch.float64)
                self._collective_round(header)
        finally:
            if self._handle is not None:
                if self.world > 1 and self._dist_ready:
                    try:
                        _dist().barrier(group=self.group)
                    except Exception:  # pragma: no cover
                        pass
                self._lib.b200_engine_sync(self._handle)
                for p in self._ipc_opened:
                    self._lib.b200_ipc_close_handle(C.c_void_p(p))
                self._ipc_opened = []
                self._lib.b200_engine_destroy(self._handle)
                self._handle = None

    def __del__(self):
        try:
            if not self._closed and self._handle is not None and self.world == 1:
                self.shutdown()
        except Exception:  # pragma: no cover
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.shutdown()


def default_inputs_from_words(model: ShardModel, words: np.ndarray):
    """theta words -> model inputs for the families shipped here."""
    from ..models.glm import GlmShards
    from ..models.linreg import LinregShards
    from ..models.ode import OdeShards

    if isinstance(model, LinregShards):
        th = words.view(np.float64).reshape(model.n_shards_total, 2)
        return th[:, 0].copy(), th[:, 1].copy()
    if isinstance(model, GlmShards):
        th = words.view(np.float32).reshape(model.n_chains, model.n_params)
        G, GP = model.n_groups, model.n_groups + model.n_features
        rows = th[0] if model.n_chains == 1 else th
        inputs = (rows[..., :G].copy(), rows[..., G:GP].copy())
        return inputs + (rows[..., GP:].copy(),) if model.n_family_params else inputs
    if isinstance(model, OdeShards):
        return model.inputs_from_words(words)
    raise FederationError(f"{type(model).__name__} must implement inputs_from_words()")
