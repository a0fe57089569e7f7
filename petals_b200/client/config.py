"""Options of the client side: where the swarm is, how to route through it, how patient to be.

Every distributed model config carries these fields (reference: src/petals/client/config.py:13-35 mixes the same names into the
HF config classes), so any of them can be given to ``from_pretrained(...)``:

    AutoDistributedModelForCausalLM.from_pretrained(path, initial_peers=["/ip4/10.0.0.1/tcp/31337"], max_retries=3)

``initial_peers`` accepts what :func:`petals_b200.parallel.swarm.resolve_swarm` understands — an in-process ``Swarm`` object or
its ``inproc://name``, a rendezvous directory shared by the processes of one box, or the address of a TCP registry in
``tcp://host:port`` / libp2p multiaddr form.
"""
from __future__ import annotations

import dataclasses
import os
from typing import Optional, Sequence, Union

from petals_b200.constants import PUBLIC_INITIAL_PEERS


def _retries_from_env() -> Optional[int]:
    """``PETALS_MAX_RETRIES=n`` caps the retries of every client in the process (CI uses it so that failures surface)."""
    raw = os.environ.get("PETALS_MAX_RETRIES", "").strip()
    return int(raw) if raw else None


DEFAULT_MAX_RETRIES = _retries_from_env()


@dataclasses.dataclass
class ClientConfig:
    # ---- where -----------------------------------------------------------------------------------------------------------
    initial_peers: Sequence[str] = tuple(PUBLIC_INITIAL_PEERS)
    dht_prefix: Optional[str] = None  # uid prefix of this model's blocks ("<prefix>.<index>"); derived from the model name if unset
    active_adapter: Optional[str] = None  # LoRA adapter the servers should apply to this client's requests

    # ---- which servers ----------------------------------------------------------------------------------------------------
    allowed_servers: Optional[Sequence[str]] = None  # only route through these peer ids ...
    blocked_servers: Optional[Sequence[str]] = None  # ... and never through these
    use_server_to_server: bool = True  # let stage i hand its output to stage i+1 directly (fused NVLink hop / rpc_push)
    pipeline_chunk_tokens: int = 512  # a step of >= 2x this many tokens over >= 2 stages is ingested as a wavefront of chunks (0: never)
    # a client running on the stages' NVLink box may join their landing-ring fabric (run_server --fabric_address ...): its inputs reach the
    # first stage and the last stage's outputs / gradients come back GPU to GPU (or through shared memory when the stages serve on CPU,
    # see fabric_device); collective: the fabric's world counts this client as one member.
    fabric_address: Optional[str] = None  # "host:port" of the box's fabric rendezvous
    fabric_rank: Optional[int] = None
    fabric_world: Optional[int] = None
    fabric_max_tokens: int = 8192
    fabric_device: Optional[str] = None  # where this member's landing rings live: None = the current CUDA device if any; "cpu" to join stages served on CPU
    show_route: Union[str, bool] = "inference"  # log the chosen chain: for inference sessions only, always (True) or never (False)
    max_pinged: int = 3  # how many candidate first-hop servers are pinged when a route is planned
    ping_timeout: float = 2

    # ---- on the wire (socket transports only; NVLink hops and in-process calls never serialise) --------------------------------------
    wire_compression: Optional[str] = None  # codec for the activations this client sends: NONE, FLOAT16, MEANSTD_16BIT, QUANTILE_8BIT, ...
    output_compression: Optional[str] = None  # codec servers are asked to answer in (overrides their --compression for this client)

    # ---- how patient --------------------------------------------------------------------------------------------------------
    connect_timeout: float = 5
    request_timeout: float = 3 * 60
    update_period: float = 60  # seconds between refreshes of the block -> servers table
    max_retries: Optional[int] = DEFAULT_MAX_RETRIES  # per call; None = keep trying
    min_backoff: float = 1  # retry delay grows from here ...
    max_backoff: float = 60  # ... to here (doubling)
    ban_timeout: float = 15  # a peer that failed is avoided for this long (doubling with repeated failures)

    daemon_startup_timeout: int = 60  # accepted for compatibility: there is no networking daemon to start
