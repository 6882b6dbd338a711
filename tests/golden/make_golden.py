"""Generates the golden fixtures in this directory by running the reference's OWN, UNMODIFIED source files
(/root/reference, imported through oracle/ref_shims.py) on seeded weights and inputs.  Runs only in the build
container (the GPU box has no /root/reference); the fixtures travel instead.

    python tests/golden/make_golden.py

Each fixture stores the config, the seed and the reference outputs (plus sub-sampled stage outputs); weights and
inputs are regenerated from the seed by oracle/weights.py when the fixture is checked.
"""

import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_shims, weights  # noqa: E402

CASES = {
    # name: (grid step deg, batch, model kwargs, seed)
    "forecaster_10deg_b2": dict(step=10, batch=2, seed=1, kw={}),
    "forecaster_5deg_b1": dict(step=5, batch=1, seed=2, kw={}),
    "forecaster_small_hidden64": dict(
        step=10, batch=3, seed=3,
        kw=dict(node_dim=64, edge_dim=64, num_blocks=3, hidden_dim_processor_node=64, hidden_dim_processor_edge=64,
                hidden_dim_decoder=32, feature_dim=10, aux_dim=4),
    ),  # fmt: skip
}
STAGE_STRIDE = 53  # stage outputs are stored for every 53rd mesh row only (keeps fixtures small)


def grid(step):
    return [(float(lat), float(lon)) for lat in range(-90, 90, step) for lon in range(0, 360, step)]


def run_forecaster(R, name, spec):
    lat_lons = grid(spec["step"])
    kw = spec["kw"]
    model = R.GraphWeatherForecaster(lat_lons, **kw).eval()
    shapes = weights.forecaster_shapes(num_h3=model.encoder.h3_nodes.shape[0], **kw)
    ref_sd = model.state_dict()
    assert list(shapes.keys()) == list(ref_sd.keys()), "state_dict key contract drifted"
    for k, v in ref_sd.items():
        assert tuple(v.shape) == tuple(shapes[k]), (k, v.shape, shapes[k])
    sd = weights.make_state_dict(shapes, spec["seed"])
    model.load_state_dict(sd)
    fdim = kw.get("feature_dim", 78) + kw.get("aux_dim", 24)
    x = weights.make_features(spec["batch"], len(lat_lons), fdim, spec["seed"])
    with torch.no_grad():
        enc_x, ei, ea = model.encoder(x)
        proc_x = model.processor(enc_x, ei, ea)
        out = model.decoder(proc_x, x[..., : model.feature_dim])
        out2 = model(x)
    assert torch.equal(out, out2)
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"),
        config=json.dumps(dict(step=spec["step"], batch=spec["batch"], seed=spec["seed"], kw=kw)),
        out=out.numpy(),
        enc_x_sub=enc_x.numpy()[::STAGE_STRIDE],
        proc_x_sub=proc_x.numpy()[::STAGE_STRIDE],
        enc_edge_index=model.encoder.graph.edge_index.numpy().astype(np.int32),
        enc_edge_attr=model.encoder.graph.edge_attr.numpy(),
        lat_edge_index_sum=np.array(model.encoder.latent_graph.edge_index.numpy().sum(axis=1)),
        lat_edge_attr_sub=model.encoder.latent_graph.edge_attr.numpy()[::STAGE_STRIDE],
        dec_edge_index_sub=model.decoder.graph.edge_index.numpy()[:, ::7].astype(np.int32),
        dec_edge_attr_sub=model.decoder.graph.edge_attr.numpy()[::7],
    )
    print(name, "out", tuple(out.shape), "mean|out|", float(out.abs().mean()))


def run_assimilator(R, name="assimilator_readme"):
    """README.md:75-90 configuration with fixed seeds."""
    rng = np.random.Generator(np.random.PCG64(7))
    obs = []
    for lat in range(-90, 90, 7):
        for lon in rng.uniform(0, 360, 100):
            obs.append((float(lat), float(lon), float(rng.uniform())))
    obs = obs + [(float(lat), float(lon), float(rng.uniform())) for lat in range(-90, 90, 45) for lon in range(0, 360, 24)]
    obs_t = torch.tensor(obs, dtype=torch.float)
    out_ll = grid(5)
    model = R.GraphWeatherAssimilator(output_lat_lons=out_ll, analysis_dim=24).eval()
    shapes = weights.forecaster_shapes(assimilator=True, output_dim=24)
    ref_sd = model.state_dict()
    assert list(shapes.keys()) == list(ref_sd.keys()), (set(shapes) ^ set(ref_sd))
    sd = weights.make_state_dict(shapes, 4)
    model.load_state_dict(sd)
    x = weights.make_features(1, len(obs), 2, 4)
    with torch.no_grad():
        out = model(x, obs_t)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), config=json.dumps(dict(seed=4, analysis_dim=24, step=5)),
                        obs=obs_t.numpy(), out=out.numpy())  # fmt: skip
    print(name, "out", tuple(out.shape), "mean|out|", float(out.abs().mean()))


def run_graphcast(R, name="graphcast_10deg_b2"):
    """graphcast/model.py GraphCast, replicated and efficient batching (the reference's own equivalence pair)."""
    lat_lons = grid(10)
    shapes = weights.forecaster_shapes(feature_dim=78, aux_dim=0, hidden_dim_decoder=256)
    sd = weights.make_state_dict(shapes, 5)
    x = weights.make_features(2, len(lat_lons), 78, 5)
    outs = {}
    for eff in (False, True):
        model = R.GraphCast(lat_lons, efficient_batching=eff).eval()
        assert list(model.state_dict().keys()) == list(shapes.keys())
        model.load_state_dict(sd)
        R.GraphCastConfig.balanced_checkpointing(model)
        with torch.no_grad():
            outs[eff] = model(x)
    print(name, "replicated vs efficient max diff", float((outs[False] - outs[True]).abs().max()))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), config=json.dumps(dict(step=10, batch=2, seed=5)),
                        out=outs[False].numpy(), out_efficient=outs[True].numpy())  # fmt: skip


def run_loss(name="loss_5deg"):
    """NormalizedMSELoss (losses.py:9-94) from the reference's own file on seeded inputs, normalize False and True."""
    import contextlib
    import io

    L = ref_shims.load_reference_losses()
    lat_lons = grid(5)
    rng = np.random.Generator(np.random.PCG64(11))
    B, N, F = 3, len(lat_lons), 78
    pred = torch.from_numpy(rng.standard_normal((B, N, F)).astype(np.float32))
    target = torch.from_numpy(rng.standard_normal((B, N, F)).astype(np.float32))
    var = rng.uniform(0.5, 2.0, F).astype(np.float32)
    vals = {}
    for normalize in (False, True):
        crit = L.NormalizedMSELoss(feature_variance=var.tolist(), lat_lons=lat_lons, normalize=normalize)
        with contextlib.redirect_stdout(io.StringIO()):  # the reference prints tensor shapes (losses.py:62-67)
            vals[normalize] = float(crit(pred, target))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), config=json.dumps(dict(step=5, batch=B, seed=11, features=F)),
                        feature_variance=var, loss_plain=np.float64(vals[False]), loss_normalized=np.float64(vals[True]))  # fmt: skip
    print(name, vals)


def run_constraints(R, name="forecaster_constraints_10deg_b2"):
    """GraphWeatherForecaster with each PhysicalConstraintLayer type (forecast.py:162-170,231-246; constraint_layer.py), the
    reference's own code.  The layer back-references the model as a sub-module, so the reference's state_dict() recurses
    without end: weights are loaded per sub-module.  A second, irregular case exercises the grid mapping's truncation
    (forecast.py:178-192): latitudes that are not evenly spaced, so two nodes share a cell and others stay empty."""
    out = {}
    lat_lons = grid(10)
    sd = weights.make_state_dict(weights.forecaster_shapes(), 6)
    x = weights.make_features(2, len(lat_lons), 102, 6)
    for ctype in ("additive", "multiplicative", "softmax"):
        model = R.GraphWeatherForecaster(lat_lons, constraint_type=ctype)  # (.eval() recurses through the layer's back-reference; no dropout anyway)
        for sub in ("encoder", "processor", "decoder"):
            getattr(model, sub).load_state_dict({k[len(sub) + 1:]: v for k, v in sd.items() if k.startswith(sub + ".")})
        with torch.no_grad():
            out[ctype] = model(x).numpy()
        print(name, ctype, "mean|out|", float(np.abs(out[ctype]).mean()))
    # mapping quirks: 4 x 6 grid whose latitudes are unevenly spaced
    lats, lons = [-80.0, -75.0, 10.0, 80.0], [0.0, 50.0, 130.0, 200.0, 290.0, 350.0]
    ll2 = [(a, b) for a in lats for b in lons]
    m2 = R.GraphWeatherForecaster(ll2, constraint_type="additive", feature_dim=4, aux_dim=0, output_dim=4)
    rng = np.random.Generator(np.random.PCG64(9))
    g = torch.from_numpy(rng.standard_normal((2, len(ll2), 3)).astype(np.float32))
    grid_t = m2.graph_to_grid(g)
    back = m2.grid_to_graph(grid_t)
    hr = torch.from_numpy(rng.standard_normal((2, len(ll2), 3)).astype(np.float32))
    lr = torch.from_numpy(rng.standard_normal((2, len(ll2), 3)).astype(np.float32))
    layer_out = {}
    for ctype in ("additive", "multiplicative", "softmax"):
        layer = R.GraphWeatherForecaster(ll2, constraint_type=ctype, feature_dim=4, aux_dim=0, output_dim=4).constraint
        with torch.no_grad():
            layer_out[ctype + "_graph"] = layer(hr, lr).numpy()  # 3D (graph) inputs
            layer_out[ctype + "_grid"] = layer(layer.model.graph_to_grid(hr), layer.model.graph_to_grid(lr)).numpy()  # 4D inputs
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"), config=json.dumps(dict(step=10, batch=2, seed=6, lats=lats, lons=lons)),
        additive=out["additive"], multiplicative=out["multiplicative"], softmax=out["softmax"],
        node_to_grid=np.array(m2.node_to_grid, dtype=np.int64), map_in=g.numpy(), map_grid=grid_t.numpy(), map_back=back.numpy(),
        hr=hr.numpy(), lr=lr.numpy(), **layer_out)  # fmt: skip


def run_init(R, name="forecaster_init_seed42"):
    """GraphWeatherForecaster's default initialisation under torch.manual_seed(42) on a 30-degree grid.  The full state_dict is
    ~31 MB, so the fixture keeps the key order, the shapes, 16 seeded values and the sha256 of the fp32 bytes of every tensor."""
    seed, step, per = 42, 30, 16
    torch.manual_seed(seed)
    sd = R.GraphWeatherForecaster(grid(step)).state_dict()
    rng = np.random.Generator(np.random.PCG64(0))
    vals = [v.detach().contiguous().numpy() for v in sd.values()]
    assert all(v.dtype == np.float32 for v in vals)
    index = np.stack([rng.integers(0, v.size, per) for v in vals])
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"), config=json.dumps(dict(seed=seed, step=step, keys=list(sd.keys()), shapes=[list(v.shape) for v in vals])),
        sample_index=index, sample=np.stack([v.reshape(-1)[i] for v, i in zip(vals, index)]),
        sha256=np.array([hashlib.sha256(v.tobytes()).hexdigest() for v in vals]))  # fmt: skip
    print(name, len(vals), "tensors", sum(v.size for v in vals), "values")


def regional_region():
    """A 0.5-degree box over western Europe plus a few scattered points (one near a pentagon): the movable domain of the test."""
    ll = [(38.0 + 0.5 * i, -12.0 + 0.5 * j) for i in range(40) for j in range(61)]
    ll += [(10.4, -54.2), (10.9, -53.7), (58.1, 10.9), (58.4, 11.3), (63.0, -20.0)]
    return ll


def run_regional(R, name="regional_europe_b2"):
    """RegionalForecaster (regional_forecast.py) with boundary nudging, default sizes, seeded weights: outputs without and with a
    global context; the state_dict key / shape contract and the graph sizes travel with the fixture."""
    lat_lons = regional_region()
    cfg = R.RegionalForecasterConfig(enable_nudging=True)
    model = R.RegionalForecaster(cfg)
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    sd = weights.make_state_dict(shapes, 21)
    model.load_state_dict(sd)
    x = weights.make_features(2, len(lat_lons), 102, 21)
    gc = weights.make_features(2, len(lat_lons), 78, 22)
    with torch.no_grad():
        out = model(x, lat_lons)
        out_n = model(x, lat_lons, global_context=gc)
    enc, _dec, lat, h3_idx = model.graph_builder(lat_lons)
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"), config=json.dumps(dict(seed=21, batch=2, keys=list(shapes.keys()), shapes=[list(v) for v in shapes.values()])),
        lat_lons=np.array(lat_lons, dtype=np.float64), out=out.numpy(), out_nudged=out_n.numpy(), h3_indices=np.array(h3_idx, dtype=np.int64),
        enc_edge_index=enc.edge_index.numpy().astype(np.int32), lat_edge_index=lat.edge_index.numpy().astype(np.int32),
        lat_edge_attr=lat.edge_attr.numpy())  # fmt: skip
    print(name, "out", tuple(out.shape), "cells", len(h3_idx), "latent edges", lat.edge_index.shape[1], "mean|out|", float(out.abs().mean()),
          "mean|nudged - out|", float((out_n - out).abs().mean()))


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count())
    R = ref_shims.load_reference()
    only = sys.argv[1:]
    if not only or "forecaster" in only:
        for n, s in CASES.items():
            run_forecaster(R, n, s)
    if not only or "assimilator" in only:
        run_assimilator(R)
    if not only or "graphcast" in only:
        run_graphcast(R)
    if not only or "loss" in only:
        run_loss()
    if not only or "constraints" in only:
        run_constraints(R)
    if not only or "regional" in only:
        run_regional(R)
    if not only or "init" in only:
        run_init(R)
