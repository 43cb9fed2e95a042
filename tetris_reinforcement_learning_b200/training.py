"""Training step and gating battles ("next" rows of the hot-path scope: the callers either side
of self-play).  Mirrors reference ai.py:1087-1220 (train_network_pytorch), :1871-1973
(load_data_and_train_model / get_data_filenames) and :1975-2114 (battle_networks).

New capability relative to the reference (BASELINE config 5): when torch.distributed is
initialised, gradients are averaged across ranks with ONE flat NCCL all-reduce per optimizer
step (the nets are 6-21 M parameters = 24-83 MB of fp32 gradients, latency-bound on NVLink,
so bucketing / overlap buys nothing)."""
import gc
import json
import os
import random

import numpy as np
import torch
from torch import nn

from .architectures import AuxBaseResNetConfig, compute_aux_targets
from .const import COLS, POLICY_SIZE, ROWS


def get_data_filenames(config):
    """Files of the newest `sets_to_train_with` data sets (ai.py:1929-1961)."""
    from .ai import highest_data_number
    max_set = highest_data_number(config)
    names = []
    for filename in os.listdir(config.data_dir):
        stem = filename.split(".")[0]
        if stem.isdigit() and int(stem) > max_set - config.sets_to_train_with:
            names.append(filename)
    if config.shuffle:
        random.shuffle(names)
    return names


def _load_set(path):
    """One data set: the reference's JSON sample list (<n>.txt) or a compact.CompactSet (<n>.npz)."""
    if path.endswith(".npz"):
        from .compact import CompactSet
        return CompactSet.load(path)
    with open(path) as f:
        return json.load(f)


def load_data(config):
    return [_load_set(f"{config.data_dir}/{f}") for f in get_data_filenames(config)]


class _CompactSelection:
    """Samples `index` of a CompactSet, expanded batch by batch on the training device."""

    def __init__(self, cset, index):
        self.cset, self.index = cset, np.asarray(index, dtype=np.int64)

    def __len__(self):
        return len(self.index)

    def batches(self, batch_size, shuffle, device):
        order = np.random.permutation(len(self.index)) if shuffle else np.arange(len(self.index))
        for lo in range(0, len(order), batch_size):
            yield self.cset.batch_tensors(self.index[order[lo:lo + batch_size]], device)


def _to_tensors(samples):
    cols = list(map(list, zip(*samples)))
    out = []
    for c in cols:
        t = torch.tensor(c)
        if t.dim() == 3 and t.shape[1] == ROWS and t.shape[2] == COLS:
            t = t.unsqueeze(1).float()
        out.append(t)
    return out


def allreduce_gradients(model):
    """Average gradients over all ranks with one flat all-reduce (no-op without a process group)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat /= dist.get_world_size()
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n


def sync_batchnorm_buffers(model):
    """Average the floating-point buffers (BatchNorm running mean / variance) over all ranks and take rank 0's
    integer buffers: after a data-parallel epoch every replica then holds the same module, buffers included."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    bufs = [b for b in model.buffers() if b.is_floating_point()]
    if bufs:
        flat = torch.cat([b.reshape(-1).float() for b in bufs])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat /= dist.get_world_size()
        off = 0
        for b in bufs:
            n = b.numel()
            b.copy_(flat[off:off + n].view_as(b).to(b.dtype))
            off += n
    for b in model.buffers():
        if not b.is_floating_point():
            dist.broadcast(b, src=0)


def _assert_same_step_count(n_batches, device):
    """Ranks with different batch counts would deadlock in the gradient all-reduce: fail loudly instead."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    lo = torch.tensor([n_batches], dtype=torch.int64, device=device)
    hi = lo.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    if int(lo) != int(hi):
        raise RuntimeError(f"data-parallel training needs the same number of batches on every rank (min {int(lo)}, max {int(hi)}): "
                           "give every rank the same number of samples")


def train_network_pytorch(config, model, samples, data_number=None, log=True):
    """AdamW on MSE(value) + CE(policy) (+ aux_weight * MSE(aux)); returns the mean losses."""
    from .ai import highest_data_number, logs_dir
    device = next(model.parameters()).device
    from .compact import CompactSet
    if isinstance(samples, CompactSet):
        samples = _CompactSelection(samples, np.arange(len(samples)))
    if isinstance(samples, _CompactSelection):
        class _Loader:   # same batches as the TensorDataset path, built on `device` from the packed records
            def __iter__(self_inner):
                return samples.batches(config.batch_size, config.shuffle, device)
        loader = _Loader()
    else:
        feats = _to_tensors(samples)
        loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(*feats), batch_size=config.batch_size,
                                             shuffle=config.shuffle)
    mse, ce = nn.MSELoss(), nn.CrossEntropyLoss()
    opt = torch.optim.AdamW(model.parameters(), lr=config.learning_rate, weight_decay=config.weight_decay)
    has_aux = isinstance(config.model_config, AuxBaseResNetConfig)
    aux_w = config.model_config.aux_weight if has_aux else 0.0
    model.train()
    tot = dict(loss=0.0, value=0.0, policy=0.0, aux=0.0)
    batches = 0
    n_samples = len(samples) if hasattr(samples, "__len__") else 0
    _assert_same_step_count((n_samples + config.batch_size - 1) // config.batch_size, device)
    for _ in range(config.epochs):
        for batch in loader:
            batch = [b.to(device) for b in batch]
            y_policy = batch.pop().reshape(-1, POLICY_SIZE).float()
            y_value = batch.pop().float()
            out = model(*batch)
            l_value = mse(out[0].reshape(-1), y_value)
            l_policy = ce(out[1].reshape(-1, POLICY_SIZE), y_policy)
            loss = l_value + l_policy
            if has_aux:
                l_aux = mse(out[2], compute_aux_targets(batch[0]))
                loss = loss + aux_w * l_aux
                tot["aux"] += l_aux.item()
            loss.backward()
            allreduce_gradients(model)
            opt.step()
            opt.zero_grad()
            tot["loss"] += loss.item(); tot["value"] += l_value.item(); tot["policy"] += l_policy.item()
            batches += 1
    sync_batchnorm_buffers(model)
    model.eval()
    avg = {k: v / max(batches, 1) for k, v in tot.items()}
    print(f"loss: {avg['loss']:>7f}  value: {avg['value']:>7f}  policy: {avg['policy']:>7f}" +
          (f"  aux: {avg['aux']:>7f}" if has_aux else ""))
    if log:
        entry = {"model_version": config.model_version,
                 "data_number": data_number if data_number is not None else highest_data_number(config),
                 "loss": avg["loss"], "value_loss": avg["value"], "policy_loss": avg["policy"], "backend": "pytorch"}
        if has_aux:
            entry["aux_loss"] = avg["aux"]
        with open(logs_dir() / "training_log.jsonl", "a") as f:
            f.write(json.dumps(entry) + "\n")
    return avg


def train_network(config, model, samples):
    if config.model != "pytorch":
        raise NotImplementedError("only model='pytorch' is implemented")
    return train_network_pytorch(config, model, samples)


def load_data_and_train_model(config, model, data=None):
    """'merge' loading: newest sets first, set of age a contributes a random decay_factor**a
    fraction of its samples (ai.py:1871-1901)."""
    if config.data_loading_style != "merge":
        raise NotImplementedError(f"data_loading_style={config.data_loading_style!r}")
    from .compact import CompactSet
    n_sets = 0
    if data is None:
        sets, fractions = [], []
        names = sorted(get_data_filenames(config), key=lambda x: int(x.split(".")[0]), reverse=True)
        for age, name in enumerate(names):
            sets.append(_load_set(f"{config.data_dir}/{name}"))
            fractions.append(config.decay_factor ** age)
        n_sets = len(names)
    else:
        n_sets = len(data)
        sets, fractions = list(data), [None] * len(data)      # None: every sample, in order (ai.py:1895)
    if sets and all(isinstance(one, CompactSet) for one in sets):
        # compact sets: the same recency-weighted sample of every set, as indices into the concatenation
        index, base = [], 0
        for one, frac in zip(sets, fractions):
            sel = range(len(one)) if frac is None else random.sample(range(len(one)), int(len(one) * frac))
            index.append(base + np.asarray(sel, dtype=np.int64))
            base += len(one)
        data = _CompactSelection(CompactSet.concatenate(sets), np.concatenate(index) if index else np.zeros(0, np.int64))
    elif any(isinstance(one, CompactSet) for one in sets):
        raise NotImplementedError("mixing JSON and compact data sets in one training run")
    else:
        data = []
        for one, frac in zip(sets, fractions):
            data.extend(one if frac is None else random.sample(one, int(len(one) * frac)))
        if config.shuffle:
            random.shuffle(data)
    print(f"Training with {len(data)} samples over {n_sets} sets with decay factor {config.decay_factor}")
    out = train_network(config, model, data)
    gc.collect()
    return out


def _check_threshold(wins, games, threshold, threshold_type):
    if threshold is None:
        return None
    if threshold_type == "more":
        if wins[0] > threshold * games:
            return True
        if wins[1] >= (1 - threshold) * games:
            return False
    elif threshold_type == "moreorequal":
        if wins[0] >= threshold * games:
            return True
        if wins[1] > (1 - threshold) * games:
            return False
    return None


def tally_battle_results(results):
    """Win counts of a gating battle from (winner, side) pairs — winner: 0 / 1 = the player that won, -1 = draw; side = the
    player network 1 controlled (game i plays side i % 2, reference ai.py:2087-2091).  Tally as ai.py:2103-2113: a draw
    is half a win for both, otherwise the win goes to the network that controlled the winning player."""
    wins = np.zeros(2, dtype=float)
    for w, s in results:
        if w == -1:
            wins += 0.5
        elif s == 0:
            wins[w] += 1
        else:
            wins[1 - w] += 1
    return wins


class DualCachedEvaluator:
    """Engine evaluator of a gating battle: two networks, each with its cached-trunk evaluator (trunk.CachedTrunkEvaluator /
    trunk_wide.CachedWideEvaluator).  Every leaf goes through ONE network, the one that owns the running search of its
    game (ai.py:2012-2016): the queued board images are split into two compact lists (one per network), each trunk
    writes its own feature cache, each heads kernel skips the other network's leaves.  Same engine contract as the
    single-network evaluators, so the whole step stays inside the engine's CUDA graph."""

    overlap_mode = "heads"
    gather_policy = True

    def __init__(self, cached_1, cached_2):
        self.c = (cached_1, cached_2)
        self.stamp = None
        self.engine = None          # set by battle_networks: the owner of a search is read from the engine's games

    def make_buffers(self, n_states, n_leaves, device, moves_cap=512):
        b = self.c[0].make_buffers(n_states, n_leaves, device, moves_cap)        # shared: what the encoder writes
        subs = []
        for c in self.c:
            sb = c.make_buffers(n_states, n_leaves, device, moves_cap)
            sb["images"] = torch.zeros((2 * n_leaves + 1, sb["images"].shape[1]), dtype=torch.bfloat16, device=device)   # + trash row
            sb["dest"] = torch.zeros(2 * n_leaves + 1, dtype=torch.int32, device=device)
            sb["opp"] = b["opp"]                   # opponent rows are the same indices in either cache
            subs.append(sb)
        b["subs"] = subs
        b["k"] = torch.arange(2 * n_leaves, device=device)
        b["rows_per_game"] = 2 * (n_states // n_leaves)
        return b

    def encode(self, b, states, leaf_state, leaf_parent, extras):
        self.c[0].encode(b, states, leaf_state, leaf_parent, extras)

    def _owner_of_games(self):
        from .state import GAME_DTYPE
        eng = self.engine
        g32 = eng.t["games"].view(torch.int32).view(eng.G, GAME_DTYPE.itemsize // 4)
        gid = g32[:, GAME_DTYPE.fields["game_id"][1] // 4]
        turn = eng.t["games"].view(eng.G, GAME_DTYPE.itemsize)[:, GAME_DTYPE.fields["turn"][1]].to(torch.int32)
        return (gid ^ turn) & 1                     # 0: network 1 searches (it plays player game_id & 1)

    def __call__(self, b, states, leaf_state, leaf_parent, extras, after_trunk=None, before_trunk=None, encoded=False,
                 search_buffers=None, join_movegen=None):
        with torch.cuda.device(extras.device):
            return self._evaluate(b, states, leaf_state, leaf_parent, extras, after_trunk, before_trunk, encoded,
                                  search_buffers, join_movegen)

    def _evaluate(self, b, states, leaf_state, leaf_parent, extras, after_trunk, before_trunk, encoded, search_buffers,
                  join_movegen):
        G = leaf_state.numel()
        if not encoded:
            self.encode(b, states, leaf_state, leaf_parent, extras)
        owner = self._owner_of_games()                                            # [G]
        k, n2 = b["k"], 2 * G
        valid = k < b["count"]
        game_of = (b["dest"].clamp(min=0) // b["rows_per_game"]).clamp(max=G - 1).long()
        owner_k = owner[game_of]
        for i, sb in enumerate(b["subs"]):
            m = valid & (owner_k == i)
            tgt = torch.where(m, torch.cumsum(m, 0) - 1, torch.full_like(k, n2))  # others land in the trash row
            sb["images"].index_copy_(0, tgt, b["images"])
            sb["dest"].index_copy_(0, tgt, b["dest"])
            sb["count"].copy_(m.sum().to(torch.int32).reshape(1))
            sb["own"].copy_(torch.where(owner == i, b["own"], torch.full_like(b["own"], -1)))
        b["count"].zero_()                          # consumed: the next step's encoder appends from zero
        if before_trunk is not None:
            before_trunk()
        for c, sb in zip(self.c, b["subs"]):
            c.trunk_step(sb, G)
        if after_trunk is not None:
            after_trunk()
        outs = []
        for c, sb in zip(self.c, b["subs"]):
            v = c.heads_step(sb, extras, G)
            outs.append((v.reshape(-1), c.policy(sb, search_buffers, join_movegen)))
        use2 = owner.bool()
        (v1, l1), (v2, l2) = outs
        return torch.where(use2, v2, v1), torch.where(use2[:, None], l2, l1)


def _battle_engine(NN_1, config_1, NN_2, config_2, n_games, seed, device, first_game_id, game_id_stride):
    """The engine of one shard of a gating battle on `device`: both networks' evaluators there, one engine sized for the
    larger of the two search budgets, the per-search settings of either side in params2.  -> (engine, params2)."""
    from .ai import _engine_for
    import copy
    from . import _native
    from .selfplay import best_evaluator, search_params_from_config

    def as_evaluator(nn_):
        if callable(nn_) and not isinstance(nn_, torch.nn.Module):
            return nn_
        with torch.cuda.device(device):
            return best_evaluator(copy.deepcopy(nn_).to(device), torch.bfloat16)

    ev1, ev2 = as_evaluator(NN_1), as_evaluator(NN_2)
    both_cached = getattr(ev1, "cached", None) is not None and getattr(ev2, "cached", None) is not None
    if both_cached:
        evaluator = lambda grids, extras: ev1(grids, extras)      # noqa: E731  (never called: the engine uses .cached)
        evaluator.cached = DualCachedEvaluator(ev1.cached, ev2.cached)
        dtype = torch.bfloat16
    else:
        def evaluator(grids, extras):      # generic evaluators (tests, unsupported nets): both on every leaf, then select
            v1, l1 = ev1(grids, extras)
            v2, l2 = ev2(grids, extras)
            use2 = evaluator.owner().bool()
            return torch.where(use2, v2.reshape(-1), v1.reshape(-1)), torch.where(use2[:, None], l2, l1)
        dtype = torch.bfloat16 if isinstance(NN_1, torch.nn.Module) else torch.float32
    # the engine is sized for the larger of the two search budgets; the per-search settings come from params2
    big = config_1 if max(config_1.playout_iterations()[0], config_1.MAX_ITER) >= max(config_2.playout_iterations()[0], config_2.MAX_ITER) \
        else config_2
    eng = _engine_for(big, evaluator, n_games, seed=seed, device=device, restart_finished=False, dtype=dtype,
                      first_game_id=first_game_id, game_id_stride=game_id_stride)
    if both_cached:
        evaluator.cached.engine = eng
    else:
        helper = DualCachedEvaluator(None, None)
        helper.engine = eng
        evaluator.owner = helper._owner_of_games
    pair = (_native.SearchParams * 2)(search_params_from_config(config_1, eng.seed, False, game_id_stride),
                                      search_params_from_config(config_2, eng.seed, False, game_id_stride))
    for p in pair:
        p.seed = eng.seed
    params2 = torch.frombuffer(bytearray(bytes(pair)), dtype=torch.uint8).to(device)
    eng.buf.params2 = params2.data_ptr()
    return eng, params2


def battle_networks(NN_1, config_1, NN_2, config_2, threshold, threshold_type, games,
                    network_1_title="Network 1", network_2_title="Network 2", screen=None, seed=None,
                    first_game_id=0, game_id_stride=1):
    """All `games` battles run concurrently on the GPU (the reference's batched variant, ai.py:2071-2114: network 1
    plays player (game index & 1), no early termination, post-hoc threshold).  Every search runs with the network AND
    the search settings (config_1 / config_2) of the side to move at the root (ai.py:2012-2016); the two configs may
    differ in anything but the ruleset.  No random opening plies (ai.py:1588-1608 is play_game only).
    first_game_id / game_id_stride shard the battles over ranks (ids first, first + stride, ...).
    config_1.engine_devices: the battles are further sharded by id over those devices (devices.shard_games), all
    engines stepped from this thread; the tallies are summed and the threshold applies to the merged tally."""
    from .ai import _time_seed
    from .devices import engine_devices, shard_games
    if config_1.ruleset != config_2.ruleset:
        raise NotImplementedError("Ruleset's aren't equal")
    seed = _time_seed(seed)      # one key for every shard
    devs = engine_devices(config_1)
    shards = [_battle_engine(NN_1, config_1, NN_2, config_2, sh["num_games"], seed, devs[sh["shard"]], sh["first_game_id"],
                             sh["game_id_stride"])
              for sh in shard_games(games, games, first_game_id, game_id_stride, len(devs))]
    ends = []
    chunk = max(8, min(config_1.MAX_ITER, config_2.MAX_ITER))
    running = [eng for eng, _ in shards]
    while running:
        for eng in running:     # queue every engine's graphs before the first drain waits for its device
            eng.step(chunk)
        for eng in running:
            ends.extend(eng.drain()[1])
            eng.check_status(ignore=0x20)        # sample records are not read here: a full sample ring is harmless
        running = [eng for eng in running if eng.get_ctl()["active"].any()]
    wins = tally_battle_results((int(e["winner"]), int(e["game_id"]) % 2) for e in ends)
    return wins, _check_threshold(wins, games, threshold, threshold_type)
