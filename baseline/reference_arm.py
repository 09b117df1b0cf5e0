"""Reference arm of the headline benchmark (``bench.py --impl reference``).

Runs the UNMODIFIED reference package that ``build()`` installs at ``oracle/_ref``
(``oracle/build_reference.py``) through its own public API and stock code path:

* one ``ArraysToArraysService(wrap_logp_grad_func(f))`` gRPC worker PROCESS per data shard
  (the reference's deployment model, ``/root/reference/demo_node.py:98-108``), placed on the
  GPU that owns the shard; ``f`` is plain PyTorch (two bf16 matmuls + elementwise) — none of
  this repository's kernels, models or engine;
* the client is the reference's ``LogpGradServiceClient`` per worker, fanned out with
  ``asyncio.gather`` exactly like its ``ParallelAsyncOp`` (``op_async.py:114-130``), results
  summed on the host.

The reference's two third-party imports that have no wheel in this offline image (betterproto,
grpclib) are satisfied by the API shims in ``baseline/shims`` (built on the installed grpcio);
the reference's own code is byte-for-byte what pip installed.  The JSON line says so.
"""
from __future__ import annotations

import asyncio
import json
import multiprocessing as mp
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
METRIC = "logp+grad evals/sec for 8-shard federated GLM"
NOTE = (
    "unmodified reference code from oracle/_ref (oracle/build_reference.py); its third-party deps betterproto/grpclib "
    "have no offline wheel and are provided as API shims over grpcio (baseline/shims); worker compute is stock "
    "PyTorch (bf16 matmuls); timing is wall clock around the client's gather (this path has no single device stream)"
)


def _paths():
    for p in (os.path.join(ROOT, "oracle", "_ref"), os.path.join(HERE, "shims")):
        if p not in sys.path:
            sys.path.insert(0, p)


def _synth(rows, features, seed, dev):
    """Same synthetic shard as the product arm (bf16 X ~ N(0,1), Bernoulli y)."""
    import torch

    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    beta_true = (torch.randn(features, generator=gen, device=dev) * 0.05).float()
    X = torch.empty(rows, features, dtype=torch.bfloat16, device=dev)
    y = torch.empty(rows, dtype=torch.float32, device=dev)
    chunk = 1 << 20
    for r0 in range(0, rows, chunk):
        r1 = min(rows, r0 + chunk)
        xb = torch.randn(r1 - r0, features, generator=gen, device=dev, dtype=torch.float32).to(torch.bfloat16)
        X[r0:r1] = xb
        p = torch.sigmoid(xb.float() @ beta_true + 0.3)
        y[r0:r1] = (torch.rand(r1 - r0, generator=gen, device=dev) < p).float()
    return X, y


def _worker(shard, port, gpu, rows, features, ready):
    _paths()
    import numpy as np
    import torch

    import grpclib.server
    from pytensor_federated import ArraysToArraysService, wrap_logp_grad_func

    if torch.cuda.is_available():
        dev = torch.device("cuda", gpu)
        torch.cuda.set_device(dev)
    else:  # plumbing tests only (B200FED_REF_ALLOW_CPU=1)
        dev = torch.device("cpu")
    X, y = _synth(rows, features, 1000 + shard, dev)

    def logp_grad(intercept, beta):
        b = torch.as_tensor(np.array(beta, dtype=np.float32), device=dev)
        eta = (X @ b.to(torch.bfloat16)).float() + float(np.asarray(intercept).reshape(-1)[0])
        ll = (y * eta - torch.nn.functional.softplus(eta)).sum()
        r = y - torch.sigmoid(eta)
        g = (r.to(torch.bfloat16) @ X).float()
        d_ic = np.asarray(intercept, dtype=np.float64) * 0 + float(r.sum())
        return np.asarray(float(ll)), [d_ic, g.cpu().numpy().astype(np.float64)]

    async def main():
        server = grpclib.server.Server([ArraysToArraysService(wrap_logp_grad_func(logp_grad))])
        await server.start("127.0.0.1", port)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        ready.set()
        await server.wait_closed()

    asyncio.new_event_loop().run_until_complete(main())


def main(args) -> None:
    _paths()
    try:
        import pytensor_federated  # noqa: F401  (the reference)
        from pytensor_federated import LogpGradServiceClient
    except Exception as ex:  # noqa: BLE001
        print(json.dumps({"impl": "reference", "unavailable": f"cannot import the reference from oracle/_ref: {ex}"}))
        return
    import numpy as np
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() and not os.environ.get("B200FED_REF_ALLOW_CPU"):
        print(json.dumps({"impl": "reference", "unavailable": "no CUDA device for the reference workers"}))
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo")

    base_port = 52000 + (int(os.environ.get("MASTER_PORT", "29500")) % 500) * 10
    ctx = mp.get_context("spawn")
    mine = [s for s in range(args.shards) if s % world == rank]
    procs, events = [], []
    for s in mine:
        ev = ctx.Event()
        p = ctx.Process(target=_worker, args=(s, base_port + s, local_rank, args.rows, args.features, ev), daemon=True)
        p.start()
        procs.append(p)
        events.append(ev)
    ok = all(ev.wait(600) for ev in events)
    line = None
    try:
        if world > 1:
            flag = torch.tensor([1 if ok else 0])
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = bool(flag.item())
        if not ok:
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "reference workers did not come up"}))
            return
        if rank == 0:
            sys.path.insert(0, ROOT)
            from bench import ClockSampler, dump_outputs  # the clock sampler and the .npy writer, nothing of the product path

            clients = [LogpGradServiceClient("127.0.0.1", base_port + s) for s in range(args.shards)]
            rng = np.random.default_rng(7)
            P = args.features
            thetas = [
                (rng.normal(size=(1,)).astype(np.float32) * 0.1, rng.normal(size=(P,)).astype(np.float32) * 0.02)
                for _ in range(args.steps + args.warmup)
            ]

            async def evaluate(theta):
                results = await asyncio.gather(*[c.evaluate_async(*theta) for c in clients])
                logp = sum(float(r[0]) for r in results)
                d_ic = sum(np.asarray(r[1][0], dtype=np.float64) for r in results)
                d_beta = sum(np.asarray(r[1][1], dtype=np.float64) for r in results)
                return logp, d_ic, d_beta

            loop = asyncio.new_event_loop()
            asyncio.set_event_loop(loop)
            for i in range(args.warmup):
                loop.run_until_complete(evaluate(thetas[i]))
            sampler = ClockSampler(local_rank).start()
            checksum = 0.0
            t0 = time.perf_counter()
            for i in range(args.steps):
                logp, d_ic, d_beta = loop.run_until_complete(evaluate(thetas[args.warmup + i]))
                checksum += logp
            elapsed = time.perf_counter() - t0
            clocks = sampler.stop()
            if getattr(args, "dump_outputs", None):
                dump_outputs(args.dump_outputs, [np.asarray(logp), d_ic, d_beta])
            value = args.steps / elapsed
            line = {
                "metric": METRIC,
                "value": value,
                "unit": "evals/s",
                "n_gpus": world,
                "steps": args.steps,
                "warmup": args.warmup,
                "ms_per_step": 1000.0 * elapsed / args.steps,
                "higher_is_better": True,
                "scaling": "strong",
                "vs_baseline": None,
                "dtype": "bf16",
                "data": "synthetic",
                "impl": "reference",
                "config": {
                    "model": "federated logistic GLM (logp + gradient)",
                    "shards": args.shards,
                    "rows_per_shard": args.rows,
                    "features": args.features,
                    "chains_per_eval": 1,
                    "global_batch": args.shards * args.rows,
                    "seq_len": args.features,
                    "parallelism": f"{args.shards} gRPC worker processes, {args.shards // world} per GPU x{world}",
                    "l2_policy": "inputs (>= 5 GB per GPU) are larger than the 126 MB L2; no flush needed",
                    "note": NOTE,
                },
                "clocks": clocks,
                "e2e": {
                    "value": value,
                    "unit": "evals/s",
                    "h2d_bytes_per_step": args.shards * (P + 1) * 4,
                    "d2h_bytes_per_step": args.shards * (P + 2) * 4,
                },
                "gpu_launches": 0,
                "checksum": checksum,
            }
            del clients
    finally:
        if world > 1:
            try:
                dist.barrier()
            except Exception:
                pass
        for p in procs:
            p.terminate()
        for p in procs:
            p.join(10)
        if world > 1:
            dist.destroy_process_group()
    if line is not None:
        out = json.dumps(line)
        print(out, flush=True)
        if getattr(args, "out", None):
            with open(args.out, "a") as fh:
                fh.write(out + "\n")
