import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


def pytest_collection_modifyitems(config, items):
    """`gpu` tests need a B200: skip them (instead of failing in CUDA initialisation) on a host without one."""
    try:
        import torch
        ok = torch.cuda.is_available() and torch.cuda.get_device_capability(0)[0] == 10
    except Exception:
        ok = False
    if ok:
        return
    skip = pytest.mark.skip(reason="needs an sm_100 (B200) GPU")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


def load_golden(name):
    """The arrays of tests/golden/<name>.npz and of its continuation files <name>.2.npz, <name>.3.npz, ...  Golden
    files are kept under 1 MB each, so a large case is spread over several; an array found in more than one of them
    is split along its first axis, in file order, and is joined here."""
    import numpy as np
    parts, k, path = {}, 1, os.path.join(GOLDEN, name + ".npz")
    while os.path.exists(path):
        with np.load(path) as g:
            for key in g.files:
                parts.setdefault(key, []).append(g[key])
        k += 1
        path = os.path.join(GOLDEN, "%s.%d.npz" % (name, k))
    if not parts:
        raise FileNotFoundError(os.path.join(GOLDEN, name + ".npz"))
    return {key: v[0] if len(v) == 1 else np.concatenate(v) for key, v in parts.items()}


def relinf(a, b):
    """max|a-b| / max|b|  (SURVEY section 7 hard part 4: the tolerance is infinity-norm relative)."""
    import numpy as np
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    denom = max(float(np.max(np.abs(b))), 1e-30)
    return float(np.max(np.abs(a - b))) / denom


def outlier_fraction(a, b, tol=1e-5):
    """Fraction of elements with |a-b| > tol * max|b|.

    Used for post-Adam tables: the first Adam steps move an element by ~lr*sign(g), so an element whose
    gradient cancels to rounding noise can legitimately land lr*2 away (SURVEY section 7, hard part 4).
    Parity is then stated as: all but a vanishing fraction of elements within tol, none further than the
    Adam step bound."""
    import numpy as np
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    denom = max(float(np.max(np.abs(b))), 1e-30)
    return float(np.mean(np.abs(a - b) > tol * denom))
