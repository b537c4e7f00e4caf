import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run by the driver with -m gpu)")
    # the native libraries are built artefacts (git-ignored): build them once if this checkout has none yet
    libs = [os.path.join(ROOT, "lt_mapper_b200", n) for n in ("libltr_b200.so", "libltr_removert.so", "ltremovert_b200")]
    libs += [os.path.join(ROOT, "oracle", "liboracle.so"), os.path.join(ROOT, "synth", "libltr_synth.so")]
    if not all(os.path.exists(p) for p in libs):
        import __graft_entry__
        __graft_entry__.build()


@pytest.fixture(scope="session")
def small_pair():
    """6-keyframe two-session synthetic pair, 32 beams x 900 steps (fast enough for the CPU oracle)."""
    import synth
    return synth.make_pair(6, beams=32, az_steps=900)


@pytest.fixture(scope="session")
def small_maps(small_pair):
    """Voxelised global maps of the small pair, built by the oracle."""
    import oracle
    out = []
    for s in small_pair:
        R = oracle.Removerter()
        R.load_session(0, s.xyzi, s.offsets, s.poses)
        R.load_session(1, s.xyzi[:0], np.zeros(1, np.int64), s.poses[:0])
        R.stage("makeGlobalMap")
        out.append(R.cloud("map_global_curr_", 0))
    return out
