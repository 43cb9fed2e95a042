"""`Config` — the drop-in configuration object (reference ai.py:62-216).

Same keyword arguments, defaults, attribute names, `copy()`, `model_dir` / `data_dir` and value
range helpers as the reference, so scripts written against `ai.Config` run unchanged.  Extra,
B200-only knobs live under `engine_*` attributes with defaults, they are not constructor
arguments of the reference and never change search semantics.
"""
import os
from pathlib import Path

from .architectures import AuxBaseResNetConfig

# Where data and models are saved: <cwd>/../Storage like the reference (ai.py:57-59), unless
# TRL_STORAGE overrides it.  Unlike the reference nothing is created at import time.
def storage_dir():
    return Path(os.environ.get("TRL_STORAGE", Path.cwd().parent / "Storage"))


_DEFAULTS = dict(
    visual=True,
    model_version=7.0, data_version=2.9,
    ruleset="s2",
    model="keras", use_tflite=True, tflite_num_threads=2, batched_inference=False,
    model_config=None,  # AuxBaseResNetConfig() per instance
    move_algorithm="convolutional",
    use_tanh=False,
    training_games=100, training_loops=1, sets_to_train_with=10, battle_games=200,
    gating_threshold=0.52, gating_threshold_type="moreorequal",
    MAX_ITER=400, CPUCT=0.75, DPUCT=1,
    FpuStrategy="reduction", FpuValue=0.1,
    use_root_softmax=True, RootSoftmaxTemp=1.1,
    temperature=0.1,
    training=False, learning_rate=0.001, weight_decay=0.0, epochs=1, batch_size=64,
    data_loading_style="merge", decay_factor=0.9, augment_data=True, shuffle=True,
    use_experimental_features=False, save_all=False, loss_weights=None,  # [1, 1] per instance
    use_random_starting_moves=False,
    use_playout_cap_randomization=True, playout_cap_chance=0.25, playout_cap_mult=5,
    use_dirichlet_noise=True, DIRICHLET_ALPHA=0.1, DIRICHLET_S=25, DIRICHLET_EXPLORATION=0.25,
    use_dirichlet_s=True,
    use_forced_playouts_and_policy_target_pruning=False, CForcedPlayout=1,
)


class Config:
    # B200-only knob (not a constructor argument of the reference): "json" = the reference's <n>.txt list of
    # 13-element samples, "compact" = <n>.npz CompactSet (compact.py), 270x smaller and expanded on the training device.
    # None = the caller's default: make_training_set writes JSON (drop-in for the reference's trainer), self_play_loop
    # (whose trainer reads both) writes compact sets; ai.export_training_set_json turns a compact set into <n>.txt.
    engine_data_format = None
    # B200-only knob: the devices generate_games / make_training_set, battle_networks, analyse / MCTS and
    # evaluate_positions run on, from one process (devices.parse_engine_devices).  None = the current device, "all" =
    # every visible device, or a list of device indices (duplicates put several engines on one device).  Games are
    # sharded by id and positions by contiguous block; the merged results equal one device's for the fused-trunk
    # networks (selfplay.best_evaluator), except evaluate_positions' policies (cuBLAS policy GEMM: one bf16 rounding),
    # and are not promised bit for bit for networks on the PyTorch / cuDNN evaluator (INTEGRATION.md section 1).
    engine_devices = None

    def __init__(self, **kwargs):
        unknown = set(kwargs) - set(_DEFAULTS)
        if unknown:
            raise TypeError(f"Config.__init__() got an unexpected keyword argument {sorted(unknown)[0]!r}")
        for name, default in _DEFAULTS.items():
            setattr(self, name, kwargs.get(name, default))
        if self.model_config is None:
            self.model_config = AuxBaseResNetConfig()
        if self.loss_weights is None:
            self.loss_weights = [1, 1]

    def copy(self):
        c = Config(**{k: getattr(self, k) for k in _DEFAULTS})
        for k, v in vars(self).items():
            if k.startswith("engine_"):
                setattr(c, k, v)
        return c

    @property
    def model_dir(self):
        sub = "pytorch_models" if self.model == "pytorch" else "models"
        return f"{storage_dir()}/{sub}/{self.ruleset}.{self.model_version}"

    @property
    def data_dir(self):
        return f"{storage_dir()}/data/{self.ruleset}.{self.data_version}"

    @property
    def value_max(self):
        return 1

    @property
    def value_mid(self):
        return 0 if self.use_tanh else 0.5

    @property
    def value_min(self):
        return -1 if self.use_tanh else 0

    def negate_value(self, value):
        return -value if self.use_tanh else 1 - value

    # playout-cap iteration counts (ai.py:323-330)
    def playout_iterations(self):
        """-> (long, short) iteration counts used when playout-cap randomisation is active."""
        import math
        denom = self.playout_cap_chance * (self.playout_cap_mult - 1) + 1
        return (math.ceil(self.playout_cap_mult * (self.MAX_ITER / denom)), math.floor(self.MAX_ITER / denom))


def config_to_dict(config):
    d = {k: getattr(config, k) for k in _DEFAULTS if k != "model_config"}
    d["model_config"] = vars(config.model_config)
    return d
