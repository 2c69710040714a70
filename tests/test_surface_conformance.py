"""The plugin surface is the reference's: ray_lightning's classes and module names, read from its source by AST
(oracle/make_surface_golden.py, stored in tests/golden/reference_surface.json), against this package's."""
import inspect
import json
import os

import pytest

REF_SURFACE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_surface.json")


@pytest.fixture(scope="module")
def ref():
    with open(REF_SURFACE) as f:
        return json.load(f)


def _mine(fn):
    """fn's signature in the stored form: [[[name, default], ...], vararg, kwarg, [kwonly, ...]]."""
    sig = inspect.signature(fn)
    pos, var, kw, kwonly = [], None, None, []
    for p in sig.parameters.values():
        if p.kind == p.VAR_POSITIONAL:
            var = p.name
        elif p.kind == p.VAR_KEYWORD:
            kw = p.name
        elif p.kind == p.KEYWORD_ONLY:
            kwonly.append(p.name)
        else:
            pos.append([p.name, None if p.default is p.empty else p.default])
    return [pos, var, kw, kwonly]


def test_ray_strategy_surface(ref):
    from ray_lightning_b200 import RayStrategy
    rm = ref["RayStrategy"]
    assert rm["__init__"] == _mine(RayStrategy.__init__)
    for name, sig in rm.items():
        assert hasattr(RayStrategy, name), name
        if name != "__init__" and not isinstance(inspect.getattr_static(RayStrategy, name), property):
            assert sig[0] == _mine(getattr(RayStrategy, name))[0], name
    assert RayStrategy.strategy_name == "ddp_ray"


def test_sharded_and_horovod_surface(ref):
    from ray_lightning_b200 import HorovodRayStrategy, RayShardedStrategy
    assert RayShardedStrategy.strategy_name == "ddp_sharded_ray"
    rm = ref["HorovodRayStrategy"]
    assert rm["__init__"] == _mine(HorovodRayStrategy.__init__)
    for name in rm:
        assert hasattr(HorovodRayStrategy, name), name
    assert HorovodRayStrategy.strategy_name == "horovod_ray"


def test_launcher_and_executor_surface(ref):
    from ray_lightning_b200.launchers import RayHorovodLauncher, RayLauncher
    from ray_lightning_b200.launchers.utils import _RayExecutorImpl, _RayOutput
    for name, sig in ref["RayLauncher"].items():
        assert hasattr(RayLauncher, name), name
        assert sig == _mine(getattr(RayLauncher, name)), name
    for name, sig in ref["RayExecutor"].items():
        assert sig == _mine(getattr(_RayExecutorImpl, name)), name
    assert list(_RayOutput._fields) == ref["_RayOutput_fields"]
    assert ref["RayHorovodLauncher"]["launch"] == _mine(RayHorovodLauncher.launch)


def test_module_level_names(ref):
    import ray_lightning_b200 as pkg
    from ray_lightning_b200 import session, tune, util
    assert sorted(pkg.__all__) == sorted(ref["__all__"])
    for mod, key in ((session, "session_names"), (util, "util_names")):
        for name in ref[key]:
            if name != "DelayedGPUAccelerator":
                assert hasattr(mod, name), (key, name)
    for name in ("TuneReportCallback", "TuneReportCheckpointCallback", "get_tune_resources", "is_session_enabled", "TUNE_INSTALLED"):
        assert hasattr(tune, name)
