"""Stand-ins for the packages the reference's driver scripts import but this image lacks, so that
`{TRAIN_FINAL,INFERENCE,INFERENCE_TIMER}.py` of a reference checkout (BUCKGNN_REFERENCE_DIR) can be
EXECUTED UNMODIFIED against this repo's `Models` package (tests/test_reference_scripts.py).  Test infrastructure only.

Stubbed: torch_geometric.loader.DataLoader / torch_geometric.data.Data (a collating loader over the synthetic
plates of buckgnn_b200.synth), torch_geometric.nn + torch_scatter (oracle/reference_source.py shims; Utils/Losses.py
imports torch_scatter), ray + ray.tune (+ .schedulers, .logger) + ray.train, matplotlib(.pyplot), and
Dataset_Preparation.GraphCreate (needs pyNastran and FE files: replaced by synthetic-graph loaders).
Loaded from the REAL reference files: Dataset_Preparation/Normalizer.py, Dataset_Preparation/Metrics.py,
Utils/Losses.py.
"""
import contextlib
import importlib.util
import sys
import types

import torch

from buckgnn_b200.synth import collate, make_plate_graph
from oracle import reference_source as RS

REF = RS.REFERENCE_DIR


class StubDataLoader:
    """torch_geometric.loader.DataLoader for a list of graphs: sequential batches, PyG `Batch` layout."""

    def __init__(self, dataset, batch_size=1, shuffle=False, **kw):
        self.dataset, self.batch_size = list(dataset), int(batch_size)

    def __len__(self):
        return -(-len(self.dataset) // self.batch_size)

    def __iter__(self):
        for i in range(0, len(self.dataset), self.batch_size):
            yield collate(self.dataset[i:i + self.batch_size])


def synthetic_dataset(n, first_index=0, **kw):
    return [make_plate_graph(first_index + i, nx=6, ny=5, **kw) for i in range(n)]


def _load_folder_dataset(data_dir, normalizer=None, **kw):
    return synthetic_dataset(6, first_index=100)


def _load_single_data(args):
    return make_plate_graph(7, nx=6, ny=5)


class _FakePool:
    def __init__(self, processes=None):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def imap(self, fn, it):
        return map(fn, it)


class _AnyAttr(types.ModuleType):
    """A module whose every attribute is a do-nothing callable / class (matplotlib, ray reporters ...)."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        class _Dummy:
            def __init__(self, *a, **k):
                pass

            def __call__(self, *a, **k):
                return self

            def __getattr__(self, n):
                return _Dummy()
        _Dummy.__name__ = name
        return _Dummy


class _NoRaySession:
    """ray.train.get_context() outside a tune session: no trial id -> TRAIN_FINAL.py:209-218 takes the manual-run branch
    (its `except RuntimeError` branch leaves `ray_running` unbound, a latent bug of the reference not exercised here)."""

    def get_trial_id(self):
        return None


def _no_ray_context():
    return _NoRaySession()


@contextlib.contextmanager
def script_environment():
    """sys.modules / sys.path as the reference scripts expect them; restored on exit."""
    saved_modules = dict(sys.modules)
    saved_path = list(sys.path)
    try:
        shim_saved = RS.install_shims()                          # torch_geometric(.nn), torch_scatter
        tg = sys.modules["torch_geometric"]
        loader = types.ModuleType("torch_geometric.loader")
        loader.DataLoader = StubDataLoader
        data = types.ModuleType("torch_geometric.data")
        data.Data = type("Data", (), {})
        tg.loader, tg.data = loader, data
        sys.modules["torch_geometric.loader"] = loader
        sys.modules["torch_geometric.data"] = data

        ray = _AnyAttr("ray")
        tune = _AnyAttr("ray.tune")
        tune.grid_search = lambda values: values[0]
        train = _AnyAttr("ray.train")
        train.get_context = _no_ray_context
        train.report = lambda *a, **k: None
        ray.tune, ray.train = tune, train
        sys.modules.update({"ray": ray, "ray.tune": tune, "ray.train": train,
                            "ray.tune.schedulers": _AnyAttr("ray.tune.schedulers"),
                            "ray.tune.logger": _AnyAttr("ray.tune.logger")})
        mpl = _AnyAttr("matplotlib")
        sys.modules.update({"matplotlib": mpl, "matplotlib.pyplot": _AnyAttr("matplotlib.pyplot")})

        # packages of the reference: real files for what is importable, a stub for the BDF/OP2 graph builder
        for pkg in ("Dataset_Preparation", "Utils"):
            m = types.ModuleType(pkg)
            m.__path__ = [f"{REF}/{pkg}"]
            sys.modules[pkg] = m
        gc = types.ModuleType("Dataset_Preparation.GraphCreate")
        gc.load_folder_dataset = _load_folder_dataset
        gc.load_single_data = _load_single_data
        sys.modules["Dataset_Preparation.GraphCreate"] = gc
        for k in [k for k in sys.modules if k == "Models" or k.startswith("Models.")]:
            del sys.modules[k]                                   # the scripts must import THIS repo's Models afresh
        yield
    finally:
        ours = ("torch_geometric", "torch_scatter", "ray", "matplotlib", "Dataset_Preparation", "Utils", "Models", "_reference_")
        for k in list(sys.modules):                 # only what this environment put there (torch lazily imports its own)
            if k.startswith(ours):
                del sys.modules[k]
                if k in saved_modules:
                    sys.modules[k] = saved_modules[k]
        sys.path[:] = saved_path


def load_script(name):
    """Executes <reference checkout>/<name>.py as a module (not as __main__), unmodified."""
    spec = importlib.util.spec_from_file_location(f"_reference_{name}", f"{REF}/{name}.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cpu_forward_through_oracle(model_cls):
    """Replacement for `BuckGNN.forward` IN TESTS ON THE CPU BOX: checks the call contract of the reference's call sites
    (`model(batch.x, batch.edge_index, batch.edge_attr, batch.batch)` -> `(pred, batch)`) and evaluates the oracle
    with the module's own parameters / buffers (functional_call), so autograd and BatchNorm updates land on them."""
    from oracle import buckgnn_oracle as O
    calls = []

    def forward(self, x, edge_index, edge_attr, batch=None, mask=None):
        assert x.dim() == 2 and x.dtype == torch.float32
        assert edge_index.dtype == torch.int64 and edge_index.shape[0] == 2
        assert edge_attr.dim() == 2 and edge_attr.shape[0] == edge_index.shape[1]
        assert batch is None or (batch.dtype == torch.int64 and batch.shape[0] == x.shape[0])
        kw = {k: v for k, v in self._ctor_kwargs.items()
              if k not in ("precision", "cta_group", "cache_index", "fold_encoder", "train_precision", "fuse_pool")}
        twin = O.OracleBuckGNN(**kw).train(self.training)
        state = dict(self.named_parameters())
        state.update(dict(self.named_buffers()))
        calls.append((self.training, tuple(x.shape)))
        return torch.func.functional_call(twin, state, (x, edge_index, edge_attr, batch))

    model_cls.forward_calls = calls
    return forward
