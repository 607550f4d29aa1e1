"""CPU-side checks: the C-ABI library loads and exports every declared symbol, the module mirror has the
reference's parameter names, reference checkpoints convert.  No compute calls (no GPU here)."""
import importlib.abc
import os
import pickle
import re
import sys
import types
import zipfile

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, load_weights


def test_library_loads_and_exports_every_declared_symbol():
    from newtonnet_b200 import _lib
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, 'include', 'newtonnet_b200.h')).read()
    declared = set(re.findall(r'^NN_API [\w\s\*]+?\b(nn_\w+)\(', hdr, flags=re.M))
    assert declared, 'no declarations parsed'
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.nn_version() >= 100
    assert lib.nn_get_gemm_backend() in (0, 1, 2)
    # struct layouts agree with the header (sizes computed independently with the C compiler rules)
    import ctypes as C
    assert C.sizeof(_lib.Mat) == 4 * 8
    assert C.sizeof(_lib.LayerWeights) == 7 * 32 + 7 * 8
    assert C.sizeof(_lib.Weights) == 8 + 2 * 8 + 8 * (7 * 32 + 7 * 8) + 2 * 32 + 6 * 8 + 3 * 32 + 4 * 8
    assert C.sizeof(_lib.Nbr) == 6 * 4 + 13 * 8 + 8
    assert C.sizeof(_lib.GemmArgs) == 10 * 8 + 5 * 4 + 4       # five int32 fields, padded to pointer alignment
    assert lib.nn_nbr_workspace_bytes(1000, 4) > 0
    assert lib.nn_eval_workspace_bytes(1000, 4, 30000, 3, 1) > lib.nn_eval_workspace_bytes(1000, 4, 30000, 3, 0)


def test_no_cpu_fallback():
    from newtonnet_b200.models import NewtonNet
    m = NewtonNet(output_properties=['energy', 'gradient_force'])
    m.eval()
    z = torch.tensor([8, 1, 1]); pos = torch.rand(3, 3); cell = torch.zeros(1, 3, 3); batch = torch.zeros(3, dtype=torch.long)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m(z, pos, cell, batch)


def test_state_dict_keys_match_reference():
    from newtonnet_b200.models import NewtonNet
    m = NewtonNet(output_properties=['energy', 'gradient_force'])
    ref = load_weights('seed0')
    sd = m.state_dict()
    assert set(sd) == set(ref)
    assert all(tuple(sd[k].shape) == ref[k].shape for k in ref)
    assert sum(v.numel() for v in sd.values()) == 401155
    # frequencies are fp32(n*pi) exactly as the reference creates them (representations.py:220)
    assert np.array_equal(sd['embedding_layers.edge_embedding.embedding.frequencies'].numpy(),
                          ref['embedding_layers.edge_embedding.embedding.frequencies'])


def test_factories_and_unsupported_heads():
    from newtonnet_b200.layers import get_activation_by_string, get_precision_by_string, get_scaler_by_string
    from newtonnet_b200.models import NewtonNet, get_aggregator_by_string, get_output_by_string
    assert isinstance(get_activation_by_string('swish'), torch.nn.SiLU)
    with pytest.raises(NotImplementedError):
        get_activation_by_string('relu')
    assert get_precision_by_string('single') is torch.float32
    with pytest.raises(ValueError):
        get_precision_by_string('bf16')
    assert get_scaler_by_string('energy').scale is not None and get_scaler_by_string('stress').scale is None
    for key in ('gradient_force', 'stress', 'virial'):
        get_output_by_string(key); get_aggregator_by_string(key)
    for key in ('charge', 'bec'):
        with pytest.raises(NotImplementedError):
            get_output_by_string(key, 128, torch.nn.SiLU())
    assert len(list(get_output_by_string('direct_force', 128, torch.nn.SiLU()).parameters())) == 6
    ln = NewtonNet(layer_norm=True, output_properties=['energy', 'gradient_force', 'direct_force'])
    assert 'interaction_layers.2.layer_norm.bias' in ln.state_dict() and 'scalers.2.scale.weight' in ln.state_dict()
    with pytest.raises(NotImplementedError):
        NewtonNet(output_properties=['charge', 'energy'])
    m = NewtonNet(output_properties=['energy', 'gradient_force'])
    assert m.embedding_layers.requires_dr is True
    m.eval()
    assert m.output_layers[1].create_graph is False
    m.train()
    assert m.output_layers[1].create_graph is True


class _ReferencePathPickler(pickle._Pickler):
    """Names this package's classes by the reference's module paths (`newtonnet.models.output.SumAggregator`, ...), as
    a checkpoint pickled by the reference itself does.  Derived from the pure-Python pickle._Pickler: the C pickler
    writes class references without calling an overridable save_global, so only this class lets every global be renamed."""

    def save_global(self, obj, name=None):
        mod = getattr(obj, '__module__', None) or ''
        if not mod.startswith('newtonnet_b200.'):
            return super().save_global(obj, name)
        self.write(pickle.GLOBAL + f'newtonnet.{mod[len("newtonnet_b200."):]}\n{obj.__qualname__}\n'.encode())
        self.memoize(obj)


_reference_path_pickle = types.ModuleType('reference_path_pickle')
_reference_path_pickle.Pickler = _ReferencePathPickler


def _write_legacy_md17_checkpoint(path, cutoff, properties):
    """A whole-module fp64 pickle in the older class layout of the reference's shipped MD17 checkpoint
    (scripts/md17_model/training_1/models/best_model.pt): top-level newtonnet.models.newtonnet.NewtonNet with
    `embedding_layer` (singular) holding `node_embedding.weight` and `edge_embedding.frequencies`, `infer_properties`
    instead of `output_properties`, `newtonnet.models.output.SumAggregator` aggregators, the MD17 weights.  The inner
    classes of `embedding_layer.edge_embedding` / `.norm` are stand-ins: the shipped file is not part of this repository."""
    from newtonnet_b200.models import NewtonNet
    from newtonnet_b200.models.output import SumAggregator
    legacy_names = {   # the shipped file's key names (tests/golden/make_golden.py, load_shipped_state_dict)
        'embedding_layers.node_embedding.weight': 'embedding_layer.node_embedding.weight',
        'embedding_layers.edge_embedding.embedding.frequencies': 'embedding_layer.edge_embedding.frequencies',
    }
    m = NewtonNet(output_properties=['energy', 'gradient_force']).double()
    emb = m._modules.pop('embedding_layers')
    emb.edge_embedding = torch.nn.Module()
    emb.edge_embedding.register_parameter('frequencies', torch.nn.Parameter(torch.zeros(20, dtype=torch.float64)))
    emb.norm = torch.nn.Module()
    emb.norm.r = cutoff
    m.embedding_layer = emb
    m.aggregators = torch.nn.ModuleList([SumAggregator() for _ in properties])
    del m.output_properties
    m.infer_properties = list(properties)
    sd = {legacy_names.get(k, k): torch.tensor(v, dtype=torch.float64) for k, v in load_weights('md17').items()}
    torch.nn.Module.load_state_dict(m, sd, strict=True)
    torch.save(m, path, pickle_module=_reference_path_pickle, pickle_protocol=2)


def _hide_reference_package(monkeypatch):
    """Neither the reference nor this repository's `newtonnet` shim importable: compat's aliases must resolve the pickle."""
    class Blocker(importlib.abc.MetaPathFinder):
        def find_spec(self, name, path=None, target=None):
            if name == 'newtonnet' or name.startswith('newtonnet.'):
                raise ImportError(f'no module named {name!r}')
            return None
    for name in [n for n in sys.modules if n == 'newtonnet' or n.startswith('newtonnet.')]:
        monkeypatch.delitem(sys.modules, name)
    monkeypatch.setattr(sys, 'meta_path', [Blocker()] + sys.meta_path)


def test_shipped_legacy_checkpoint_loads(tmp_path, monkeypatch):
    from newtonnet_b200.compat import load_model
    w = load_weights('md17')
    path = tmp_path / 'best_model.pt'
    _write_legacy_md17_checkpoint(path, 5.0, ['energy', 'gradient_force'])
    with zipfile.ZipFile(path) as zf:
        skeleton = zf.read(next(n for n in zf.namelist() if n.endswith('/data.pkl')))
    assert b'newtonnet.models.output\nSumAggregator\n' in skeleton and b'newtonnet.models.newtonnet\nNewtonNet\n' in skeleton
    assert b'newtonnet_b200' not in skeleton

    def check(m, cutoff, properties):
        assert m.output_properties == properties and m.cutoff == cutoff
        sd = m.state_dict()
        assert set(sd) == set(w)
        assert all(np.array_equal(sd[k].float().numpy(), w[k]) for k in w)

    check(load_model(str(path), map_location='cpu'), 5.0, ['energy', 'gradient_force'])     # through the `newtonnet` shim
    # cutoff and heads are read from the pickle, not defaulted
    _write_legacy_md17_checkpoint(tmp_path / 'other.pt', 4.5, ['energy'])
    check(load_model(str(tmp_path / 'other.pt'), map_location='cpu'), 4.5, ['energy'])
    _hide_reference_package(monkeypatch)
    check(load_model(str(path), map_location='cpu'), 5.0, ['energy', 'gradient_force'])     # through compat's aliases
    assert 'newtonnet' not in sys.modules


def test_pickled_mirror_module_round_trip(tmp_path):
    """A whole-module pickle (the reference's checkpoint format, trainer.py:219) of the mirror loads back."""
    from newtonnet_b200.compat import load_model, model_from_state_dict
    w = load_weights('seed0')
    m = model_from_state_dict({k: torch.tensor(v) for k, v in w.items()})
    p = tmp_path / 'model.pt'
    torch.save(m, p)
    m2 = load_model(str(p), map_location='cpu')
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    torch.save(m.state_dict(), p)
    m3 = load_model(str(p), map_location='cpu')
    assert set(m3.state_dict()) == set(w)


def test_struct_layout_of_dd_comm_matches_header(tmp_path):
    """nn_dd_comm is filled from Python: its ctypes mirror must have the C compiler's size and field offsets."""
    import ctypes as C
    import subprocess
    from newtonnet_b200 import _lib
    src = tmp_path / 'sz.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu %%zu %%zu %%zu\\n", '
                   'sizeof(nn_dd_comm), offsetof(nn_dd_comm, landing), offsetof(nn_dd_comm, peer_landing), offsetof(nn_dd_comm, send_idx), '
                   'offsetof(nn_dd_comm, step), offsetof(nn_dd_comm, peer_flags));return 0;}\n' % os.path.join(ROOT, 'include', 'newtonnet_b200.h'))
    exe = tmp_path / 'sz'
    subprocess.run(['gcc', str(src), '-o', str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    D = _lib.DDComm
    assert got == [C.sizeof(D), D.landing.offset, D.peer_landing.offset, D.send_idx.offset, D.step.offset, D.peer_flags.offset]


def test_reference_import_paths_resolve_to_this_package():
    """The `newtonnet` shim: reference-side import lines work unchanged (scripts/simulate.py:6, scripts/newtonnet_train.py:9,
    utils/ase_interface.py:8-13) and resolve to the CUDA-backed classes."""
    import importlib
    import newtonnet_b200
    nn_pkg = importlib.import_module('newtonnet')
    assert getattr(nn_pkg, '__backend__', None) == 'newtonnet_b200', 'a different `newtonnet` package shadows the shim'
    from newtonnet.models import NewtonNet
    from newtonnet.models.newtonnet import EmbeddingNet, InteractionNet
    from newtonnet.models.output import DerivativeProperty, SecondDerivativeProperty, get_aggregator_by_string, get_output_by_string
    from newtonnet.layers.precision import get_precision_by_string
    from newtonnet.layers.scalers import get_scaler_by_string, set_scaler_by_string, ScaleShift
    from newtonnet.layers.representations import EdgeEmbedding
    from newtonnet.data import RadiusGraph
    from newtonnet.utils.ase_interface import MLAseCalculator
    from newtonnet.utils.pretrained_models import download_checkpoint
    assert NewtonNet is newtonnet_b200.models.NewtonNet
    assert MLAseCalculator is importlib.import_module('newtonnet_b200.utils.ase_interface').MLAseCalculator
    m = NewtonNet(output_properties=['energy', 'gradient_force'])
    assert type(m).__module__ == 'newtonnet_b200.models.newtonnet' and isinstance(m.embedding_layers, EmbeddingNet)
    with pytest.raises(ImportError):
        from newtonnet.data import MolecularDataset   # noqa: F401


def test_whole_module_pickle_of_current_reference_loads_without_les():
    """Pickle written by the unmodified reference (tests/golden/make_pickle_golden.py): class paths newtonnet.* and a
    `les.Les` instance inside aggregators.0 - `les` is not installed here (advisor finding, round 1)."""
    import importlib.util
    from newtonnet_b200.compat import load_model
    from newtonnet_b200.models import NewtonNet
    assert importlib.util.find_spec('les') is None
    model = load_model(os.path.join(GOLDEN, 'ref_module_pickle.pt'), map_location='cpu')
    assert isinstance(model, NewtonNet) and model.output_properties == ['energy', 'gradient_force']
    assert len(model.interaction_layers) == 1
    sd = model.state_dict()
    assert not any(k.startswith('aggregators.') for k in sd)
    assert all(torch.isfinite(v).all() for v in sd.values())
    assert float(sd['scalers.0.shift.weight'].abs().sum()) > 0      # the randomised scaler made it through


def test_activation_of_a_pickled_module_is_not_silently_replaced():
    from newtonnet_b200.compat import _activation_name, load_model
    from newtonnet_b200.models import NewtonNet
    m = NewtonNet(output_properties=['energy'])
    assert _activation_name(m) == 'swish'
    for layer in m.interaction_layers:
        layer.message_nodepart[1] = torch.nn.ReLU()
    with pytest.raises(NotImplementedError):
        load_model(_as_plain_module(m))


def _as_plain_module(m):
    """A torch.nn.Module that is not this package's NewtonNet but has its module tree (like a reference pickle)."""
    class Foreign(torch.nn.Module):
        pass
    f = Foreign()
    f.__dict__.update(m.__dict__)
    return f


def test_weight_gradient_routing_modes_nest_and_restore():
    """newtonnet_b200.train: 'skip' while the forces are derived (no X^T dY formed), restored on exit, also when nested or
    when the body raises; routing itself needs no GPU."""
    import torch
    from newtonnet_b200 import train
    assert train._weight_grad_mode == 'autograd'
    W = torch.nn.Parameter(torch.zeros(128, 128))
    with train._skip_weight_grads():
        assert train._weight_grad_mode == 'skip'
        assert train._weight_grad(W, torch.zeros(4, 128), torch.zeros(4, 128)) is None      # nothing launched
        with train._skip_weight_grads():
            assert train._weight_grad_mode == 'skip'
        assert train._weight_grad_mode == 'skip'
    assert train._weight_grad_mode == 'autograd'
    try:
        with train._skip_weight_grads():
            raise KeyError('x')
    except KeyError:
        pass
    assert train._weight_grad_mode == 'autograd'
