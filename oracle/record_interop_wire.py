"""Records the gRPC messages that ``tests/test_reference_interop.py`` replays.

Usage: ``python oracle/record_interop_wire.py PATH_TO_PYTENSOR_FEDERATED_CHECKOUT``

The upstream ``pytensor-federated`` package is not part of this repository, so the interop tests do not
run it.  This script runs it once (its missing third-party imports betterproto / grpclib are provided
by ``baseline/shims``) behind a byte-logging gRPC proxy and writes what went over the wire to
``tests/golden/reference_wire.json``:

* ``product_client``: this package's client against the upstream server -- the requests the client
  sent and the upstream server's answers (``Evaluate`` / ``EvaluateStream`` / ``GetLoad``);
* ``reference_client``: the upstream client against the upstream server serving the product of its
  inputs -- the upstream client's requests and the upstream server's answers.

Messages are stored as hex strings of their serialized bytes.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
import textwrap
import time
from concurrent import futures

import grpc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from _helpers import free_port  # noqa: E402

from pytensor_federated_b200.rpc import ROUTE_EVALUATE, ROUTE_EVALUATE_STREAM, ROUTE_GET_LOAD  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_wire.json")

UPSTREAM_SERVER = textwrap.dedent(
    """
    import asyncio, sys
    import numpy as np
    import grpclib.server
    from pytensor_federated import ArraysToArraysService, wrap_logp_grad_func

    def logp_grad(a, b):
        return np.asarray(-(a - 1.0) ** 2 - np.sum((b + 2.0) ** 2)), [np.asarray(-2 * (a - 1.0)), -2 * (b + 2.0)]

    def product(*inputs):
        return (np.prod(inputs),)

    async def main(port, which):
        func = wrap_logp_grad_func(logp_grad) if which == "logp_grad" else product
        server = grpclib.server.Server([ArraysToArraysService(func)])
        await server.start("127.0.0.1", port)
        print("READY", flush=True)
        await server.wait_closed()

    asyncio.new_event_loop().run_until_complete(main(int(sys.argv[1]), sys.argv[2]))
    """
)

UPSTREAM_CLIENT = textwrap.dedent(
    """
    import sys
    import numpy as np
    from pytensor_federated import ArraysToArraysServiceClient
    client = ArraysToArraysServiceClient("127.0.0.1", int(sys.argv[1]))
    out = client.evaluate(np.array(6), np.array(7))
    assert out[0] == 42, out
    out = client.evaluate(np.array(1.5), np.array(4.0), use_stream=False)
    assert float(out[0]) == 6.0, out
    print("OK", flush=True)
    """
)


class LoggingProxy(grpc.GenericRpcHandler):
    """Forwards the three routes byte for byte to ``upstream`` and logs every message."""

    def __init__(self, upstream_port: int):
        self.channel = grpc.insecure_channel(f"127.0.0.1:{upstream_port}")
        self.log = []

    def _unary(self, route):
        call = self.channel.unary_unary(route)

        def handler(request, context):
            response = call(request)
            self.log.append({"route": route, "request": request.hex(), "response": response.hex()})
            return response

        return grpc.unary_unary_rpc_method_handler(handler)

    def _stream(self, route):
        call = self.channel.stream_stream(route)

        def handler(requests, context):
            sent = []

            def tap():
                for r in requests:
                    sent.append(r)
                    yield r

            for response in call(tap()):
                self.log.append({"route": route, "request": sent[-1].hex(), "response": response.hex()})
                yield response

        return grpc.stream_stream_rpc_method_handler(handler)

    def service(self, handler_call_details):
        route = handler_call_details.method
        if route == ROUTE_EVALUATE_STREAM:
            return self._stream(route)
        if route in (ROUTE_EVALUATE, ROUTE_GET_LOAD):
            return self._unary(route)
        return None


def _upstream_env(reference: str):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "baseline", "shims"), reference, ROOT])
    return env


def _record(reference: str, which: str, client) -> list:
    port = free_port()
    upstream = subprocess.Popen([sys.executable, "-c", UPSTREAM_SERVER, str(port), which], env=_upstream_env(reference),
                                stdout=subprocess.PIPE, text=True)
    proxy = LoggingProxy(port)
    server = grpc.server(futures.ThreadPoolExecutor(max_workers=8), handlers=[proxy])
    proxy_port = server.add_insecure_port("127.0.0.1:0")
    server.start()
    try:
        assert upstream.stdout.readline().strip() == "READY"
        client(proxy_port)
        time.sleep(0.5)
        return list(proxy.log)
    finally:
        server.stop(1)
        upstream.terminate()
        upstream.wait(10)


def product_client(port: int) -> None:
    import numpy as np

    from pytensor_federated_b200 import LogpGradServiceClient, service

    client = LogpGradServiceClient("127.0.0.1", port)
    client.evaluate(np.array(3.0), np.array([0.0, 1.0]))
    service.get_useful_event_loop().run_until_complete(service.get_load_async("127.0.0.1", port))
    del client


def main(reference: str) -> None:
    def upstream_client(port: int) -> None:
        res = subprocess.run([sys.executable, "-c", UPSTREAM_CLIENT, str(port)], env=_upstream_env(reference),
                             capture_output=True, text=True, timeout=120)
        assert res.returncode == 0 and "OK" in res.stdout, res.stderr[-2000:]

    golden = {
        "product_client": _record(reference, "logp_grad", product_client),
        "reference_client": _record(reference, "product", upstream_client),
    }
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as fh:
        json.dump(golden, fh, indent=1)
        fh.write("\n")
    print(f"wrote {OUT}: " + ", ".join(f"{k}: {len(v)} messages" for k, v in golden.items()))


if __name__ == "__main__":
    main(os.path.abspath(sys.argv[1]))
