"""The C-ABI shared library loads and exports every symbol include/gw_b200.h declares (no compute without a GPU),
and the host-side modules keep the reference's state_dict contract."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

import __graft_entry__ as ge
from graph_weather_b200 import _capi


@pytest.fixture(scope="module", autouse=True)
def _built():
    ge.build()


def test_library_exports_header_symbols():
    lib = _capi.load()
    syms = _capi.header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), s
    assert lib.gw_abi_version() == 1
    assert [lib.gw_timing_tag_name(i).decode() for i in range(lib.gw_timing_num_tags())][:3] == ["const", "enc_grid", "enc_mesh"]


def test_no_cpu_path():
    """The product path must fail loudly instead of computing on the host."""
    from graph_weather_b200 import GraphWeatherForecaster

    ll = [(float(a), float(b)) for a in range(-90, 90, 30) for b in range(0, 360, 30)]
    m = GraphWeatherForecaster(ll)
    with pytest.raises(RuntimeError, match="no CPU"):
        m(torch.randn(1, len(ll), 102))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            _capi.Plan("cuda:0", n_in=1, n_out=1, n_mesh=1, n_lat_edges=1, n_dec_edges=1, in_dim=1, enc_edge_attr_dim=2, out_dim=1,
                       residual_dim=0, node_dim=8, edge_dim=8, hidden_node=8, hidden_edge=8, hidden_layers_node=2,
                       hidden_layers_edge=2, hidden_dec=8, hidden_layers_dec=2, num_blocks=1, precision=0, max_batch=1)  # fmt: skip


def test_state_dict_contract_matches_oracle_shapes():
    from graph_weather_b200 import GraphWeatherAssimilator, GraphWeatherForecaster
    from oracle import weights

    ll = [(float(a), float(b)) for a in range(-90, 90, 30) for b in range(0, 360, 30)]
    m = GraphWeatherForecaster(ll)
    sd = m.state_dict()
    shapes = weights.forecaster_shapes()
    assert list(sd.keys()) == list(shapes.keys())
    assert all(tuple(sd[k].shape) == tuple(shapes[k]) for k in sd)
    a = GraphWeatherAssimilator(output_lat_lons=ll, analysis_dim=24)
    shapes = weights.forecaster_shapes(assimilator=True, output_dim=24)
    assert list(a.state_dict().keys()) == list(shapes.keys())
    # the key the survey quotes as part of the drop-in contract
    assert tuple(sd["processor.graph_processor.blocks.3.edge_model.edge_mlp.model.0.weight"].shape) == (256, 768)


def test_same_seed_same_init_as_reference(golden_dir):
    """Under the same seed the default initialisation is the reference's, bit for bit.  The fixture holds the reference's
    key order, shapes, a seeded sample of values and the sha256 of every tensor (tests/golden/make_golden.py::run_init)."""
    from graph_weather_b200 import GraphWeatherForecaster

    z = np.load(os.path.join(golden_dir, "forecaster_init_seed42.npz"))
    cfg = json.loads(str(z["config"]))
    ll = [(float(a), float(b)) for a in range(-90, 90, cfg["step"]) for b in range(0, 360, cfg["step"])]
    torch.manual_seed(cfg["seed"])
    mine = GraphWeatherForecaster(ll).state_dict()
    assert list(mine.keys()) == cfg["keys"]
    for i, k in enumerate(cfg["keys"]):
        v = mine[k].detach().contiguous().numpy()
        assert v.dtype == np.float32 and list(v.shape) == cfg["shapes"][i], k
        np.testing.assert_array_equal(v.reshape(-1)[z["sample_index"][i]], z["sample"][i], err_msg=k)
        assert hashlib.sha256(v.tobytes()).hexdigest() == str(z["sha256"][i]), k


def test_graphcast_wrapper_contract():
    from graph_weather_b200 import GraphCast, GraphCastConfig
    from oracle import weights

    ll = [(float(a), float(b)) for a in range(-90, 90, 30) for b in range(0, 360, 30)]
    m = GraphCast(ll, efficient_batching=True)
    shapes = weights.forecaster_shapes(feature_dim=78, aux_dim=0, hidden_dim_decoder=256)
    assert list(m.state_dict().keys()) == list(shapes.keys())
    GraphCastConfig.balanced_checkpointing(m)
    assert (m._checkpoint_encoder, m._checkpoint_processor_segments, m._checkpoint_decoder) == (True, -1, True)
    GraphCastConfig.full_checkpointing(m)
    assert m._checkpoint_model and not m._checkpoint_encoder


def test_perm16_feature_order_contract():
    """The weight packing (csrc/gw_pack.cu, perm16_f) and the chain kernel (csrc/gw_tc3.cu) agree on this map: inside every group
    of 16 features, packed position a holds logical feature f(a) = 4*((a>>1)&3) + 2*(a>>3) + (a&1).  It must be a permutation,
    and the four accumulator columns a tcgen05.ld.16x256b.x2 fragment gives lane t -- 2t, 2t+1, 8+2t, 9+2t (t = lane % 4) -- must
    be four consecutive logical features starting at 4t, which is what makes the 128-bit global accesses of the epilogue legal."""

    def f(a):
        return (a & ~15) | (4 * ((a >> 1) & 3) + 2 * ((a >> 3) & 1) + (a & 1))

    assert sorted(f(a) for a in range(64)) == list(range(64))
    for group in (0, 16, 32):
        for t in range(4):
            cols = [group + 2 * t, group + 2 * t + 1, group + 8 + 2 * t, group + 9 + 2 * t]
            assert [f(c) for c in cols] == [group + 4 * t + i for i in range(4)]
    src = open(os.path.join(ge.ROOT, "graph_weather_b200", "csrc", "gw_pack.cu")).read()
    assert "(4 * ((a >> 1) & 3) + 2 * ((a >> 3) & 1) + (a & 1))" in src  # the formula the test restates
