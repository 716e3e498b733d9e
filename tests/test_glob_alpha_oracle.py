"""CPU: the attention weights of the reference's global-feature runs.  tests/golden_glob/*.pt hold the last layer's
`stored_alpha` and the filtered edge list, minted by the reference's own `GNN`; the oracle (which stores alpha from the
full feature rows, global channels included) reproduces both bit for bit, so the GPU read-out can be checked against
the oracle wherever no fixture exists."""
import copy

import pytest
import torch

import gad_testutil as util
from oracle import gnn_oracle
from test_glob_features import NAMES, _dataset, _load


@pytest.mark.parametrize("name", NAMES)
def test_oracle_reproduces_reference_alpha_with_global_features(name):
    fx = _load(name)
    opt, data, md = util.fixture_opt(fx), util.fixture_batch(fx), fx["mesh_dims_list"][0]
    ref = gnn_oracle.GNNRef(_dataset(md), copy.deepcopy(opt))
    ref.load_state_dict(fx["state_dict"], strict=True)
    ref.train()
    out, _, ei = ref(data, return_states=True)
    assert torch.equal(out, fx["x_phys"])
    assert torch.equal(ei, fx["edge_index_filtered"])
    alpha = ref.conv_layers[-1].stored_alpha
    assert alpha.shape == fx["alpha_last"].shape
    assert torch.equal(alpha, fx["alpha_last"])
