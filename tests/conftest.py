import os
import sys
import tarfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs /root/reference (build container only)")


def _extract(name, tmp_path_factory):
    d = tmp_path_factory.mktemp(name.replace(".tar.gz", ""))
    with tarfile.open(os.path.join(GOLDEN, name)) as tf:
        tf.extractall(d)
    return str(d)


@pytest.fixture(scope="session")
def sample_dir(tmp_path_factory):
    """two real frames of the reference's data/mg_tfsi_dme (timesteps 0 and 2500000)"""
    return _extract("sample_frames.tar.gz", tmp_path_factory)


@pytest.fixture(scope="session")
def c1_dir(tmp_path_factory):
    """config C1 at full length: all 101 frames of the reference's data/mg_tfsi_dme, columns id type x y z xu yu zu
    (oracle/make_c1_fixture.py; 24 MB, too large to commit, so git-ignored and absent from a fresh clone)"""
    path = os.path.join(ROOT, "tests", "golden_large", "c1_frames.tar.gz")
    if not os.path.exists(path):
        pytest.skip("tests/golden_large/c1_frames.tar.gz is absent (oracle/make_c1_fixture.py builds it from a checkout of the "
                    "reference project named by MDPROP_REFERENCE_ROOT)")
    d = tmp_path_factory.mktemp("c1_frames")
    with tarfile.open(path) as tf:
        tf.extractall(d)
    return str(d)


@pytest.fixture(scope="session")
def mini_dir(tmp_path_factory):
    return _extract("mini_traj.tar.gz", tmp_path_factory)


@pytest.fixture(scope="session")
def visc_dir(tmp_path_factory):
    return _extract("visc_log.tar.gz", tmp_path_factory)


@pytest.fixture(scope="session")
def water_dir(tmp_path_factory):
    return _extract("water_box.tar.gz", tmp_path_factory)


@pytest.fixture(scope="session")
def slab_dir(tmp_path_factory):
    """surface slab + two-species fluid, 2 frames (oracle/gen_golden.py make_slab_box)"""
    return _extract("slab_box.tar.gz", tmp_path_factory)


@pytest.fixture(scope="session")
def gold_density():
    import numpy as np
    return np.load(os.path.join(GOLDEN, "ref_number_density.npz"), allow_pickle=False)


@pytest.fixture(scope="session")
def gold_structural():
    import numpy as np
    return np.load(os.path.join(GOLDEN, "ref_structural.npz"), allow_pickle=False)


@pytest.fixture(scope="session")
def gold_dynamical():
    import numpy as np
    return np.load(os.path.join(GOLDEN, "ref_dynamical.npz"), allow_pickle=False)


@pytest.fixture(scope="session")
def gold_hydration():
    import numpy as np
    return np.load(os.path.join(GOLDEN, "ref_hydration.npz"), allow_pickle=False)


MASS = [16.0, 12.01, 1.008, 14.01, 32.06, 16.0, 12.01, 19.0, 24.305]
NUM_MOLS = [591, 66, 33]
NUM_ATOMS = [16, 15, 1]
ELEMENTS = ["O", "C", "H", "N", "S", "O", "C", "F", "Mg"]
