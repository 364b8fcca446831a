import importlib.util
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _import_repository_package():
    """The repository root is a package as well (ComfyUI loads it through its ``__init__.py``), so pytest collects it as
    one and imports it by its directory name through the parent directory.  That import fails, and with it every test,
    when the parent directory may be entered but not listed.  Importing the package here from its own path leaves pytest
    a module to find in ``sys.modules``; its relative import of the inner package gets the copy the tests use."""
    import comfyui_parallelanything_b200
    name = os.path.basename(ROOT)
    if (not name.isidentifier() or name in sys.modules
            or os.path.isfile(os.path.join(os.path.dirname(ROOT), "__init__.py"))):
        return                      # pytest names or finds the root package without a listing of the parent
    sys.modules[name + ".comfyui_parallelanything_b200"] = comfyui_parallelanything_b200
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "__init__.py"),
                                                  submodule_search_locations=[ROOT])
    module = importlib.util.module_from_spec(spec)
    sys.modules[name] = module
    spec.loader.exec_module(module)


_import_repository_package()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on a B200 via gpurun)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 CUDA devices")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        have = torch.cuda.is_available()
        ngpu = torch.cuda.device_count() if have else 0
    except Exception:
        have, ngpu = False, 0
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    skip_multi = pytest.mark.skip(reason="needs >= 2 CUDA devices")
    for item in items:
        if "gpu" in item.keywords and not have:
            item.add_marker(skip_gpu)
        if "multigpu" in item.keywords and ngpu < 2:
            item.add_marker(skip_multi)
