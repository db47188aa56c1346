import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
ASSET = os.path.join(ROOT, "mujoco_panda_pnp_b200", "assets", "panda_shelf_kinematic.xml")
NEUTRAL = np.array([0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79])


def tree_fk(tree, q):
    """EE-site position from a canonical KinematicTree (test helper: the product has no CPU FK)."""
    p, r = np.zeros(3), np.eye(3)
    for i in range(7):
        p = p + r @ tree.link_pos[i]
        r = r @ tree.link_rot[i]
        a = float(q[i]) - tree.qref[i]
        c, s = np.cos(a), np.sin(a)
        r = r @ np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    return p + r @ tree.ee_pos


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch

        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if have_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_fk():
    return np.load(os.path.join(GOLDEN, "fk_jac_golden.npz"))


@pytest.fixture(scope="session")
def golden_ik():
    return np.load(os.path.join(GOLDEN, "ik_reference_golden.npz"))


@pytest.fixture(scope="session")
def golden_reward():
    return np.load(os.path.join(GOLDEN, "reward_reference_golden.npz"))


@pytest.fixture(scope="session")
def oracle_model():
    from oracle import mj_oracle

    return mj_oracle.MjModel.from_xml_path(ASSET)


@pytest.fixture(scope="session")
def oracle_chain(oracle_model):
    from oracle import c_oracle

    c_oracle.build()
    return c_oracle.chain_from_model(oracle_model)


@pytest.fixture(scope="session")
def kin_model():
    from mujoco_panda_pnp_b200 import KinematicModel

    return KinematicModel.from_xml_path(ASSET)


@pytest.fixture(scope="session")
def cuda_lib():
    """Build (if needed) and load libpnp_b200.so; GPU tests call through it."""
    from mujoco_panda_pnp_b200 import _lib
    from mujoco_panda_pnp_b200.csrc import build as cuda_build

    if not os.path.exists(_lib.LIB_PATH):
        cuda_build.build()
    return _lib.load()
