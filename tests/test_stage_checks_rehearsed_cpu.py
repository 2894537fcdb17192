"""CPU: the stage checks of the gated GPU suite (tests/test_gpu_raft.py: RAFT, image propagation, flow completion — same code, same
tolerances) rehearsed on the hybrid runtime: fp16 storage, the real ProPainter kernels from their source (tests/hybrid_rt.py), numpy for the
tensor-core convolutions.  A check that cannot pass here (an API slip in the test, a tolerance below fp16 noise) would burn GPU minutes in
the first session of round 2; one that passes here still has the tensor-core convs to meet on the device."""
import os

import pytest

from conftest import ROOT

DIR = os.path.join(ROOT, "weights", "propainter")
pytestmark = pytest.mark.slow


def _needs(name):
    return pytest.mark.skipif(not os.path.exists(os.path.join(DIR, name)), reason=f"{name} not staged under weights/propainter")


@pytest.fixture(scope="module")
def hybrid():
    from hybrid_rt import HybridRuntime
    from pp_op_cases import load_emu_library
    from vsr_b200 import _capi

    lib = load_emu_library()
    saved, _capi._lib = _capi._lib, lib
    yield lambda: HybridRuntime(lib)
    _capi._lib = saved


@_needs("raft-things.pth")
def test_raft_stage_check(hybrid):
    import test_gpu_raft as G

    G.check_raft_flows(hybrid())


def test_image_propagation_stage_check(hybrid):
    import test_gpu_raft as G

    G.check_image_propagation(hybrid())


@_needs("recurrent_flow_completion.pth")
def test_flow_completion_stage_check(hybrid):
    import test_gpu_raft as G

    G.check_flow_completion(hybrid())
