"""The reference's OWN trainers, unmodified, driving this package's modules (north star: "drop-in").

What the trainers contribute - the QAT trainer's reset period and epoch length, the FSPTQ trainer's target selection,
model-state switch and per-name learning rates - is stored in tests/golden/reference_trainers.json, so both tests run
without an upstream checkout and check this package against those values.  When DLMCQ_REFERENCE_ROOT names an upstream
checkout, the fixture imports the real trainer classes, every stored value is re-derived from them and must match,
and the FSPTQ trainer's change_model_state is run on this package's modules (that one check needs the upstream code).
No compute happens here (no GPU): what is checked is the wiring the trainers rely on - class identity through
`compat.install()`, `reset_qparams` discovery and period, fnmatch name filters, `change_quant_state`,
`generate_optimizer`'s parameter groups, target selection of the block reconstruction."""
import copy
import importlib
import json
import logging
import os
import sys
import types
from fnmatch import fnmatch

import pytest
import torch
from torch import nn

REF = os.environ.get("DLMCQ_REFERENCE_ROOT", "")
HAVE_REF = bool(REF) and os.path.isdir(os.path.join(REF, "trainer"))
with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_trainers.json")) as _f:
    GOLDEN = json.load(_f)

CFG = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 8, "signed": True, "ch_axis": 0}},
       "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 8, "signed": False}},
       "exclude_layers": [], "override_options": [], "momentum": 0.1}


@pytest.fixture()
def reference_trainers():
    """Import trainer/{quantization_aware_training,fsptq}_trainer.py from the reference tree with `dlmc.*` resolved
    to this package and the reference's heavyweight side modules (tensorboard writer, yaml utils) stubbed.
    (None, None) without an upstream checkout: the tests then use the stored values."""
    import dlmc_quant_b200.compat as compat
    saved_modules = dict(sys.modules)
    saved_path = list(sys.path)
    compat.install(force=True)
    try:
        yield _import_reference_trainers() if HAVE_REF else (None, None)
    finally:
        sys.path[:] = saved_path
        mine = ("dlmc.", "trainer", "utils", "logger", "base", "matplotlib", "ruamel")
        for k in list(sys.modules):
            if k not in saved_modules and (k == "dlmc" or k.startswith(mine)):
                del sys.modules[k]
        for k in ("utils", "logger", "base"):
            if k in saved_modules:
                sys.modules[k] = saved_modules[k]
            else:
                sys.modules.pop(k, None)
        for k, v in saved_modules.items():
            if k == "trainer" or k.startswith("trainer."):
                sys.modules[k] = v


def _import_reference_trainers():
    sys.path.insert(0, REF)
    for name in ("matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    # utils.MetricTracker / logger.TensorboardWriter: stand-ins with the surface the trainers use (the reference's own
    # MetricTracker writes into read-only pandas views and fails on current pandas)
    util = types.ModuleType("utils")

    class MetricTracker:
        def __init__(self, *keys):
            self.keys = keys
        def reset(self): pass
        def reset_batch(self): pass
        def update(self, *a, **k): pass
        def result(self): return {}
        def avg(self, k): return 0.0
        def avg_batch(self, k): return 0.0
    util.MetricTracker = MetricTracker
    sys.modules["utils"] = util
    lg = types.ModuleType("logger")

    class TensorboardWriter:
        def __init__(self, *a, **k): pass
        def set_step(self, *a, **k): pass
        def add_scalar(self, *a, **k): pass
    lg.TensorboardWriter = TensorboardWriter
    sys.modules["logger"] = lg
    for k in [k for k in sys.modules if k == "trainer" or k.startswith("trainer.")]:
        del sys.modules[k]                                # e.g. the oracle shim's namespace stubs from earlier tests
    tr = types.ModuleType("trainer")
    tr.__path__ = [os.path.join(REF, "trainer")]          # bypass trainer/__init__.py (imports a missing file)
    sys.modules["trainer"] = tr
    qat = importlib.import_module("trainer.quantization_aware_training_trainer")
    fsp = importlib.import_module("trainer.fsptq_trainer")
    return qat, fsp


class _Config(dict):
    """The slice of parse_config.ConfigParser that BaseTrainer touches."""
    resume = None

    def __init__(self, tmp, **trainer):
        super().__init__(trainer={"epochs": 1, "verbosity": 2, "save_to_disk": False, "monitor": "off", **trainer},
                         grad_clip_param=0)
        self.save_dir = self.log_dir = tmp

    def get_logger(self, name, verbosity=2):
        return logging.getLogger(name)


class Net(nn.Module):
    def __init__(self):
        super().__init__()
        self.conv1 = nn.Conv2d(3, 8, 3, padding=1)
        self.block = nn.Sequential(nn.Conv2d(8, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, 8, 3, padding=1))
        self.linear = nn.Linear(8, 10)

    def forward(self, x):
        return self.linear(self.block(self.conv1(x)).mean((2, 3)))


def _loader():
    return [(torch.zeros(2, 3, 8, 8), torch.zeros(2, dtype=torch.long)) for _ in range(4)]


def test_qat_trainer_finds_and_drives_our_modules(reference_trainers, tmp_path, monkeypatch):
    qat, _ = reference_trainers
    gold = GOLDEN["qat"]
    from dlmc.utils.quantize import quantize_model           # resolves to dlmc_quant_b200.quantize
    from dlmc_quant_b200.scalar.modules.base import QBase
    net = Net()
    quantize_model(net, copy.deepcopy(CFG), None)
    assert all(isinstance(m, QBase) for m in (net.conv1, net.block[0], net.linear))
    opt = torch.optim.SGD(net.parameters(), lr=0.1)
    loader = _loader()
    assert len(loader) == gold["loader_batches"]
    period, len_epoch, model = gold["update_qparams_period"], gold["len_epoch"], net
    if qat is not None:
        monkeypatch.setattr(qat.QATTrainer, "_save_checkpoint", lambda self, epoch: None, raising=False)
        t = qat.QATTrainer(net, nn.CrossEntropyLoss(), [], opt, _Config(str(tmp_path), **gold["trainer_config"]),
                           loader, train_log_density=1, valid_log_density=1, rank=-1, world_size=-1)
        assert (t.update_qparams_period, t.len_epoch) == (period, len_epoch)
        model = t.model
    # the trainer's reset hook: `if hasattr(m, 'reset_qparams'): m.reset_qparams()` (qat_trainer.py:44-48)
    for m in net.modules():
        if isinstance(m, QBase):
            m._host_init = {"in": True, "wt": True}
            m.in_init_state.fill_(1); m.wt_init_state.fill_(1)

    def _reset(m):
        if hasattr(m, "reset_qparams"):
            m.reset_qparams()
    model.apply(_reset)
    assert all(m._host_init == {"in": False, "wt": False} and float(m.in_init_state) == 0
               for m in net.modules() if isinstance(m, QBase))
    # steps at which the trainer resets: (epoch*len + batch) % period == 1
    assert [b for b in range(4) if (1 * len_epoch + b) % period == 1] == [1, 3]
    # the parameter-name filters it logs by (qat_trainer.py:92,139) find our parameters
    names = [n for n, _ in net.named_parameters()]
    assert sum(fnmatch(n, "*in_scale*") for n in names) == 4 and all(p.requires_grad for p in net.parameters())
    # the optimizer built BEFORE the first forward holds the per-channel scale Parameters for good
    held = {id(p) for g in opt.param_groups for p in g["params"]}
    assert all(id(m.wt_scale) in held and tuple(m.wt_scale.shape)[0] == m.weight.shape[0]
               for m in net.modules() if isinstance(m, QBase))


def test_fsptq_trainer_sees_our_blocks_and_param_groups(reference_trainers, tmp_path, monkeypatch):
    _, fsp = reference_trainers
    gold = GOLDEN["fsptq"]
    from dlmc.utils.quantize import quantize_model
    from dlmc_quant_b200.recon import FSPTQReconstructor
    from dlmc_quant_b200.scalar.FSPTQuant.base import FSPTQBase
    # the class fsptq_trainer.py:9 imports by its full upstream path: one class object on both sides of the alias
    assert importlib.import_module("dlmc.quantization.scalar.FSPTQuant.base").FSPTQBase is FSPTQBase
    net, fp = Net(), Net()
    quantize_model(net, copy.deepcopy(CFG), None, quantization_type="FSPTQ")
    block_types = tuple(getattr(nn, n) for n in gold["block_dict"])
    assert [n for n, _, _ in FSPTQReconstructor(net, fp, block_types=block_types).targets()] == gold["targets"]
    # generate_optimizer (fsptq_trainer.py:136-152): our parameter names fall into the groups the reference's own
    # modules fall into - `.endswith("scales")` matches neither `in_scale` nor `wt_scale` there either, so scales train
    # at 1e-5 like weights; recon.py reproduces exactly that by default (scale_lr=None)
    ours, _ = FSPTQReconstructor(net, fp, epochs=10).generate_optimizer(net.block)
    ours_lrs = [[n, g["lr"]] for (n, _), g in zip(net.block.named_parameters(), ours.param_groups)]
    assert len(ours.param_groups) == len(gold["block_optimizer_lrs"]) and ours_lrs == gold["block_optimizer_lrs"]
    tuned, _ = FSPTQReconstructor(net, fp, epochs=10, scale_lr=1e-3).generate_optimizer(net.block)
    got = {n: g["lr"] for (n, _), g in zip(net.block.named_parameters(), tuned.param_groups)}
    assert got["0.in_scale"] == 1e-3 and got["0.wt_scale"] == 1e-3 and got["0.weight"] == 1e-5
    if fsp is None:
        return
    # the live upstream trainer: every stored value above is re-derived from it
    assert fsp.FSPTQBase is FSPTQBase
    monkeypatch.setattr(fsp.FSPTQTrainer, "_save_checkpoint", lambda self, epoch: None, raising=False)
    t = fsp.FSPTQTrainer(net, fp, None, [], None, _Config(str(tmp_path), epochs=10), _loader(),
                         block_dict={b: True for b in block_types}, train_log_density=1, valid_log_density=1, rank=-1,
                         world_size=-1)
    # target selection of train() (fsptq_trainer.py:44-59): FSPTQ layers named conv1 / linear, and block types
    picked = [n for (n, m), _ in zip(net.named_modules(), fp.modules())
              if (isinstance(m, fsp.FSPTQBase) and n in ["conv1", "linear"]) or type(m) in t.block_dict]
    assert picked == gold["targets"]
    # change_model_state (fsptq_trainer.py:155-161): conv1 keeps its input un-quantised
    t.change_model_state(net, True, True)
    for name, state in gold["change_model_state_wt_act_true"].items():
        assert {k: bool(getattr(net.get_submodule(name), k)) for k in state} == state, name
    opt, _ = t.generate_optimizer(net.block)
    ref_lrs = [[n, g["lr"]] for (n, _), g in zip(net.block.named_parameters(), opt.param_groups)]
    assert len(opt.param_groups) == len(gold["block_optimizer_lrs"]) and ref_lrs == gold["block_optimizer_lrs"]
