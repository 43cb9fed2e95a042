"""Which CUDA devices the public entry points use (`Config.engine_devices`) and how their work is split over them.

Self-play, gating battles and analysis need no collective to use several devices of one box: every random draw is keyed
by (seed, game id, purpose, search no.), so games sharded by id and merged give the set one device plays; positions
split into contiguous blocks come back in input order.  The functions here are the arithmetic of those splits; they
do not touch a device.
"""
import numbers


def parse_engine_devices(spec, n_visible, current):
    """Config.engine_devices -> list of device indices.

    None: [current] (one device, the current one); "all": every visible device; a list or tuple of indices
    (duplicates allowed: several engines share a device).  Anything else raises ValueError."""
    if spec is None:
        return [int(current)]
    if isinstance(spec, str):
        if spec != "all":
            raise ValueError(f"engine_devices must be None, 'all' or a list of device indices, not {spec!r}")
        if n_visible < 1:
            raise ValueError("engine_devices='all': no CUDA device is visible")
        return list(range(n_visible))
    if not isinstance(spec, (list, tuple)) or not spec:
        raise ValueError(f"engine_devices must be None, 'all' or a non-empty list of device indices, not {spec!r}")
    out = []
    for d in spec:
        if isinstance(d, bool) or not isinstance(d, numbers.Integral):
            raise ValueError(f"engine_devices: {d!r} is not a device index")
        if not 0 <= int(d) < n_visible:
            raise ValueError(f"engine_devices: device {int(d)} is not one of the {n_visible} visible devices")
        out.append(int(d))
    return out


def engine_devices(config):
    """The torch devices `config` runs its engines on (Config.engine_devices, resolved against the visible devices)."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("the engines need a CUDA device: the search, rules and placements run in libtrl_b200.so "
                           "(there is no CPU fallback)")
    idx = parse_engine_devices(getattr(config, "engine_devices", None), torch.cuda.device_count(),
                               torch.cuda.current_device())
    return [torch.device("cuda", d) for d in idx]


def split_evenly(n, parts):
    """n items over `parts` shares as evenly as possible, the first shares taking the remainder:
    share k = ceil((n - k) / parts), the number of i < n with i % parts == k."""
    n, parts = int(n), int(parts)
    if n < 0 or parts < 1:
        raise ValueError("split_evenly needs n >= 0 and parts >= 1")
    return [n // parts + (k < n % parts) for k in range(parts)]


def shard_games(num_games, concurrent, first_game_id, game_id_stride, n_shards):
    """Game-id shards of one call of generate_games / battle_networks over `n_shards` engines.

    Shard k plays ids first_game_id + k * game_id_stride + j * (game_id_stride * n_shards), j = 0, 1, ...: its share of
    num_games (split_evenly), with its share of `concurrent` games at a time (at least one when it has games).  The
    shards' ids are disjoint and their union is the ids one engine with (first_game_id, game_id_stride) plays, so a
    caller's own rank sharding (first_game_id = rank, game_id_stride = world) composes with this one.
    -> [dict(first_game_id, game_id_stride, num_games, concurrent)], shards without games left out."""
    stride = int(game_id_stride) * int(n_shards)
    out = []
    for k, (n_k, c_k) in enumerate(zip(split_evenly(num_games, n_shards), split_evenly(concurrent, n_shards))):
        if n_k:
            out.append({"shard": k, "first_game_id": int(first_game_id) + k * int(game_id_stride), "game_id_stride": stride,
                        "num_games": n_k, "concurrent": max(1, c_k)})
    return out


def contiguous_blocks(n, parts):
    """Positions 0 .. n-1 as `parts` contiguous blocks of split_evenly sizes -> [(lo, hi)], empty blocks included."""
    out, lo = [], 0
    for size in split_evenly(n, parts):
        out.append((lo, lo + size))
        lo += size
    return out
