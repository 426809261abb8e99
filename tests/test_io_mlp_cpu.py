"""CPU checks of the encoder / decoder kernel switch: its parsing and default, the models' state_dict and pickling with it on, and
that it refuses to run without CUDA (no silent fallback to the torch MLPs)."""
import pickle

import pytest
import torch

from conftest import GoldenCase
from hgn_b200 import _cabi, config
from hgn_b200 import util as hutil
from hgn_b200.migration.meshgraphnet import MeshGraphNet


@pytest.fixture
def switch():
    saved = config._io_kernels
    yield config
    config._io_kernels = saved


def _model(name="mgn_sum_L2"):
    case = GoldenCase(name)
    m = MeshGraphNet(3, 128, 2, case.meta["aggregation"], case.meta["steps"], case.meta["architecture"], case.meta["edge_sets"])
    m.load_state_dict(case.weights())
    return case, m


@pytest.mark.parametrize("text,value", [("", False), ("0", False), ("off", False), ("False", False), ("no", False),
                                        ("1", True), ("on", True), ("TRUE", True), (" yes ", True)])
def test_switch_parsing(switch, text, value):
    switch._io_kernels = text
    assert switch.io_kernels() is value


def test_switch_default_and_setter(switch):
    import os
    import subprocess
    import sys
    from conftest import ROOT
    env = {k: v for k, v in os.environ.items() if k != "HGN_B200_IO_KERNELS"}
    env["PYTHONPATH"] = os.path.join(ROOT, "hyper-graph-nets_b200")
    run = subprocess.run([sys.executable, "-c", "import hgn_b200; print(hgn_b200.io_kernels())"], env=env, capture_output=True, text=True)
    assert run.returncode == 0 and run.stdout.strip() == "False", run.stderr
    import hgn_b200
    hgn_b200.set_io_kernels(True)
    assert hgn_b200.io_kernels() is True
    hgn_b200.set_io_kernels(False)
    assert hgn_b200.io_kernels() is False
    switch._io_kernels = "maybe"
    with pytest.raises(ValueError):
        switch.io_kernels()
    m = MeshGraphNet(3, 128, 2, "sum", 1, "none", ["mesh_edges"])
    assert m.encoder.kernels is None and m.decoder.kernels is None
    assert m.encoder.precision is None and m.decoder.precision is None


def test_state_dict_unchanged_with_switch_on(switch):
    case, m_off = _model()
    switch.set_io_kernels(True)
    _, m_on = _model()
    m_on.encoder.kernels = m_on.decoder.kernels = True
    assert list(m_on.state_dict().keys()) == list(m_off.state_dict().keys()) == list(case.meta["shapes"].keys())


def test_pickled_model_carries_no_packed_cache():
    _, m = _model()
    m.encoder.kernels = m.decoder.kernels = True
    m.encoder.__dict__["_hgn_packed"] = {"node_model": {"x": object()}}
    m.decoder.__dict__["_hgn_packed"] = {"x": object()}
    m2 = pickle.loads(pickle.dumps(m))
    assert "_hgn_packed" not in m2.encoder.__dict__ and "_hgn_packed" not in m2.decoder.__dict__
    assert m2.encoder.kernels is True and m2.decoder.kernels is True
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_switch_on_without_cuda_raises(switch):
    case, m = _model()
    m.processor.precision = m.encoder.precision = m.decoder.precision = "bf16"
    switch.set_io_kernels(True)
    g = case.graph(hutil.MultiGraph, hutil.EdgeSet)
    with pytest.raises(_cabi.HgnError):
        m.encoder(g)
    with pytest.raises(_cabi.HgnError):
        m.decoder(g._replace(node_features=torch.zeros(4, 128)))


def test_switch_ignored_in_fp32_parity_mode(switch):
    """Parity mode keeps the torch MLPs whatever the switch says: on the CPU the encoder and decoder then run as before."""
    case, m = _model()
    switch.set_io_kernels(True)
    m.encoder.precision = m.decoder.precision = "fp32"
    g = case.graph(hutil.MultiGraph, hutil.EdgeSet)
    latent = m.encoder(g)
    assert latent.node_features[0].dtype == torch.float32
    out = m.decoder(latent._replace(node_features=torch.zeros(5, 128)))
    assert out.shape == (5, 3) and out.dtype == torch.float32
