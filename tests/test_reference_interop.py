"""Wire compatibility with the upstream ``pytensor-federated`` package (CPU).

``tests/golden/reference_wire.json`` holds the gRPC messages exchanged with the unmodified upstream
package, recorded by ``oracle/record_interop_wire.py``.  The upstream server is replayed from it to this
package's client, and the upstream client's requests are sent to this package's server, whose answers
must be the upstream server's answers (the ``uuid`` field identifies a call and is compared per call).
The requests recorded from this package's client are a snapshot of its own output that the upstream server
accepted; comparing with them guards against the client's encoding drifting, not against upstream.
"""
import json
import os
from concurrent import futures

import grpc
import numpy as np
import pytest

from _helpers import ServerProcess

from pytensor_federated_b200 import _pb
from pytensor_federated_b200.rpc import ROUTE_EVALUATE, ROUTE_EVALUATE_STREAM, ROUTE_GET_LOAD, OutputArrays

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "tests", "golden", "reference_wire.json")) as _fh:
    GOLDEN = json.load(_fh)

pytestmark = pytest.mark.timeout(180)


def _split(message: bytes):
    """``(items, uuid)`` of an Input/OutputArrays message, items as their serialized bytes."""
    items, uuid = [], ""
    for field, _, value in _pb.iter_fields(message):
        if field == 1:
            items.append(bytes(value))
        elif field == 2:
            uuid = bytes(value).decode("utf-8")
    return items, uuid


def _with_uuid(message: bytes, uuid: str) -> bytes:
    items, _ = _split(message)
    return b"".join(_pb.enc_len_field(1, i) for i in items) + _pb.enc_len_field(2, uuid.encode("utf-8"))


class ReplayedReferenceServer(grpc.GenericRpcHandler):
    """Answers every call with the recorded upstream answer; keeps the requests it received."""

    def __init__(self, recorded):
        self.answers = {m["route"]: bytes.fromhex(m["response"]) for m in recorded}
        self.requests = []

    def _answer(self, route, request: bytes) -> bytes:
        self.requests.append((route, request))
        if route == ROUTE_GET_LOAD:
            return self.answers[route]
        return _with_uuid(self.answers[route], _split(request)[1])

    def service(self, handler_call_details):
        route = handler_call_details.method
        if route == ROUTE_EVALUATE_STREAM and route in self.answers:
            return grpc.stream_stream_rpc_method_handler(lambda reqs, ctx: (self._answer(route, r) for r in reqs))
        if route in self.answers:
            return grpc.unary_unary_rpc_method_handler(lambda req, ctx: self._answer(route, req))
        return None


def test_product_client_talks_to_reference_server():
    from pytensor_federated_b200 import LogpGradServiceClient, service

    recorded = GOLDEN["product_client"]
    replay = ReplayedReferenceServer(recorded)
    server = grpc.server(futures.ThreadPoolExecutor(max_workers=4), handlers=[replay])
    port = server.add_insecure_port("127.0.0.1:0")
    server.start()
    try:
        client = LogpGradServiceClient("127.0.0.1", port)
        logp, (da, db) = client.evaluate(np.array(3.0), np.array([0.0, 1.0]))
        assert logp == -(2.0**2) - (4.0 + 9.0)
        assert da == -4.0
        np.testing.assert_array_equal(db, [-4.0, -6.0])
        load = service.get_useful_event_loop().run_until_complete(service.get_load_async("127.0.0.1", port))
        assert load.n_clients == 1 and 0 < load.percent_ram < 100
        del client
    finally:
        server.stop(1)
    # the client still sends what the upstream server was recorded to accept
    assert [(route, _split(req)[0]) for route, req in replay.requests] == [
        (m["route"], _split(bytes.fromhex(m["request"]))[0]) for m in recorded
    ]


def test_reference_client_talks_to_product_server():
    recorded = GOLDEN["reference_client"]
    assert [m["route"] for m in recorded] == [ROUTE_EVALUATE_STREAM, ROUTE_EVALUATE]
    with ServerProcess() as server, grpc.insecure_channel(f"127.0.0.1:{server.port}") as channel:
        stream_req, unary_req = (bytes.fromhex(m["request"]) for m in recorded)
        answers = list(channel.stream_stream(ROUTE_EVALUATE_STREAM)(iter([stream_req]), timeout=60))
        answers.append(channel.unary_unary(ROUTE_EVALUATE)(unary_req, timeout=60))
    for m, answer in zip(recorded, answers):
        want_items, _ = _split(bytes.fromhex(m["response"]))
        got_items, got_uuid = _split(answer)
        assert got_uuid == _split(bytes.fromhex(m["request"]))[1]
        assert got_items == want_items, m["route"]
    assert OutputArrays.FromString(answers[0]).arrays[0] == 42
    assert float(OutputArrays.FromString(answers[1]).arrays[0]) == 6.0
