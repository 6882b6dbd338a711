"""bench.py -- forward steps/s of GraphWeatherForecaster(lat_lons)(features), the reference's README call (README.md:48-58).

    python bench.py                                                  # BASELINE configs[1]: 1 deg, 102->78, batch 8, default path
    python bench.py --grid 0.25deg --batch 4 --precision bf16        # BASELINE configs[2]
    python bench.py --impl reference --steps 2 --warmup 1            # the reference's CPU forward on the host cores
    python bench.py --dump-outputs DIR                               # also writes the last timed step's forecast to DIR
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N [--grid 0.25deg --batch 4 --precision bf16]

The model is built exactly as a user of the reference builds it -- `GraphWeatherForecaster(lat_lons)`, no extra keyword --
unless --precision names a non-default arithmetic mode.  One step = one model(features) call at `--batch` samples per GPU;
`value` is the whole-job aggregate (steps per second summed over ranks; weak scaling).  With N > 1 every step ends at the
loss boundary (SURVEY.md 8(e)): `--boundary gather` (default) all-gathers the outputs -- issued on a side stream so that it
overlaps the next step's forward -- and `--boundary loss` exchanges the fused loss scalar instead.

The JSON line carries the contract keys plus
  roofline      the dominant kernel class by device time, timed live with CUDA events on the launching stream
                (libgwb200's gw_timing_*), algorithmic FLOPs (SURVEY.md 8(d)) / time vs the measured dense bf16 peak
  parity        max |GPU - oracle| of one sample of THIS run's output (1 deg grid; the oracle is the CPU restatement)
  cpu_baseline  the reference forward on this box's host cores, bounded sample (rank 0, N = 1 only)
  e2e           the same metric through the public module call with pinned-host inputs copied in and the forecast copied out
"""

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H_MESH, EL = 5882, 41162
FIN, FOUT = 102, 78
# per-row Linear FLOPs (2*MACs), SURVEY.md section 8
F_EDGE_MLP = 2 * (768 * 256 + 256 * 256 + 256 * 256)
F_NODE_MLP = 2 * (512 * 256 + 256 * 256 + 256 * 256)
F_NODE_ENC = 2 * (FIN * 256 + 256 * 256 + 256 * 256)
F_NODE_DEC = 2 * (256 * 128 + 128 * 128 + 128 * FOUT)


def grid_1deg():
    return [(float(lat), float(lon)) for lat in range(-90, 90) for lon in range(0, 360)]  # README.md:48-51


def grid_quarter_deg():
    """ERA5 0.25 degree grid, 721 x 1440 (SURVEY.md 8(d)): lat = -90 + 0.25 i, lon = 0.25 j."""
    lat = -90.0 + 0.25 * np.arange(721)
    lon = 0.25 * np.arange(1440)
    return np.stack(np.meshgrid(lat, lon, indexing="ij"), axis=-1).reshape(-1, 2)


GRIDS = {"1deg": grid_1deg, "0.25deg": grid_quarter_deg}
DUMP_BYTES = 48 * 2**20  # --dump-outputs writes at most this much data (under 64 MB with the .npy headers)


def output_sample(y):
    """Host copy of what one step returned, for --dump-outputs.  A forecast [B, N, F] is kept whole when it fits DUMP_BYTES,
    else at a fixed sorted sample of grid points (PCG64 seed 0, the same points for every sample); a loss is kept as is."""
    y = y.detach()
    if y.dim() != 3:
        return {"loss": y.double().cpu().numpy()}
    b, n, f = y.shape
    k = min(n, DUMP_BYTES // (b * f * 4))
    if k < n:
        idx = np.sort(np.random.Generator(np.random.PCG64(0)).choice(n, k, replace=False))
        y = y[:, torch.from_numpy(idx).to(y.device)]
    return {"forecast": y.float().cpu().numpy()}


def algorithmic_flops(n, ed):
    """F_alg per sample and per kernel class (live outputs, unfactored Linear FLOPs; SURVEY.md 8(d))."""
    per = {
        "enc_grid": n * (F_NODE_ENC + F_EDGE_MLP),
        "enc_mesh": H_MESH * F_NODE_MLP,
        "proc_p": 0.0,  # its products are layer 1 of the edge MLP, counted under proc_edge
        "proc_edge": 9 * EL * F_EDGE_MLP,
        "proc_node": 9 * H_MESH * F_NODE_MLP,
        "dec_p": 0.0,
        "dec_edge": ed * F_EDGE_MLP,
        "dec_node": n * (F_NODE_MLP + F_NODE_DEC),
    }
    return sum(per.values()), per


def source_hash():
    """Hash of the chain kernel's sources (the kernel classes profiles/traffic.json holds ncu dram bytes for): the figure is only
    quoted for the build it was measured on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "graph_weather_b200", "csrc")
    for f in ("gw_tc3.cu", "gw_tc_ptx.cuh", "gw_pack.cu"):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)  # fmt: skip
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(index):
    """Pins this process (and the pinned host buffers it is about to allocate) to the CPUs NVML reports as local to the GPU,
    so that the H2D / D2H copies of the end-to-end loop do not cross sockets.  Best effort."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def reference_model_and_inputs(lat_lons, batch, seed=42):
    """The CPU leg's model: the reference's own unmodified modules (oracle/ref_shims.py) when /root/reference exists (build
    container), else the oracle port (oracle/restate.py; GPU box).  Default initialisation under the seed the reference tests
    use; `run(x)` is one forward."""
    from oracle import ref_shims, restate

    x = None
    if ref_shims.available():
        R = ref_shims.load_reference()
        torch.manual_seed(seed)
        model = R.GraphWeatherForecaster([tuple(p) for p in np.asarray(lat_lons).tolist()]).eval()
        x = torch.randn(batch, len(lat_lons), FIN)

        def run(inp):
            with torch.no_grad():
                return model(inp)

        return "ref_shims", run, x
    from graph_weather_b200 import GraphWeatherForecaster

    torch.manual_seed(seed)
    ours = GraphWeatherForecaster(lat_lons)  # same init as the reference under the same seed (tests/test_capi.py)
    sd = {k: v.detach().clone() for k, v in ours.state_dict().items()}
    g = oracle_graphs(ours)
    x = torch.randn(batch, len(lat_lons), FIN)

    def run(inp):
        return restate.forecaster_forward(sd, g, inp)

    return "port", run, x


def oracle_graphs(model):
    e, m, d = model.encoder._g_enc, model.encoder._g_lat, model.decoder._g_dec
    return dict(enc_edge_index=torch.from_numpy(e.edge_index), enc_edge_attr=torch.from_numpy(e.edge_attr),
                lat_edge_index=torch.from_numpy(m.edge_index), lat_edge_attr=torch.from_numpy(m.edge_attr),
                dec_edge_index=torch.from_numpy(d.edge_index), dec_edge_attr=torch.from_numpy(d.edge_attr),
                num_latlons=model.encoder.num_latlons, num_h3=m.num_h3)  # fmt: skip


def pick_threads(run, x1):
    """All logical cores or one thread per physical core, whichever runs a one-sample forward faster."""
    cores = os.cpu_count()
    best_n, best_t = cores, None
    for n in sorted({cores, max(1, cores // 2)}, reverse=True):
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        run(x1)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_n, best_t = n, dt
    torch.set_num_threads(best_n)
    return best_n, best_t


def time_cpu_forward(lat_lons, step_batch, sample_batch, steps, warmup, budget_s):
    """Times `run` on `sample_batch` of the step's `step_batch` samples.  The number of timed forwards is cut so that the leg
    stays inside `budget_s` seconds; what actually ran is returned."""
    kind, run, x = reference_model_and_inputs(lat_lons, sample_batch)
    cores, t1 = pick_threads(run, x[:1])
    est = t1 * sample_batch
    did_w = 0
    for _ in range(warmup):
        if did_w >= 1 and est * (did_w + 1) > 0.3 * budget_s:
            break
        t0 = time.perf_counter()
        run(x)
        est = time.perf_counter() - t0
        did_w += 1
    ts = []
    for _ in range(max(1, steps)):
        if ts and (sum(ts) + est) > budget_s:
            break
        t0 = time.perf_counter()
        run(x)
        ts.append(time.perf_counter() - t0)
        est = ts[-1]
    t = sum(ts) / len(ts)
    return dict(kind=kind, cores=cores, seconds_per_forward=t, steps=len(ts), warmup=did_w, steps_per_s=(sample_batch / t) / step_batch)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--grid", default="1deg", choices=sorted(GRIDS))
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (default: 8 at 1 deg, 4 at 0.25 deg = BASELINE configs[1], [2])")
    ap.add_argument("--precision", default=None, choices=["auto", "fp32", "fp32_simt", "bf16"],
                    help="default: auto at 1 deg (the constructor default: fp32-faithful tcgen05), bf16 at 0.25 deg (configs[2])")  # fmt: skip
    ap.add_argument("--boundary", default="gather", choices=["gather", "gather_sync", "loss"], help="what crosses GPUs at the loss boundary (N > 1)")
    ap.add_argument("--gather-mode", default="auto", choices=["auto", "fused", "fused_peer", "p2p_copy", "nccl"],
                    help="transport of the gather boundary: fused into the forecast's last kernel (NVLink multicast / peer stores), copy engines, or NCCL")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the oracle comparison of this run's output")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (float32 forecast, "
                    "sampled at fixed grid points above 48 MiB; float64 loss with --boundary loss) to compare two builds")  # fmt: skip
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if a.batch is None:
        a.batch = 8 if a.grid == "1deg" else 4
    if a.precision is None:
        a.precision = "auto" if a.grid == "1deg" else "bf16"

    # stdout carries exactly one JSON line: anything libraries print in between (NCCL's version banner comes from C code)
    # is sent to stderr by pointing file descriptor 1 there until the line is written
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    lat_lons = GRIDS[a.grid]()
    n_pts = len(lat_lons)
    cfg = {"workload": None, "grid": {"1deg": "1deg lat -90..89 x lon 0..359 (README.md:48-51)", "0.25deg": "0.25deg ERA5 721 x 1440"}[a.grid],
           "points": n_pts, "batch_per_gpu": a.batch, "global_batch": a.batch * world, "hidden": 256, "processor_blocks": 9,
           "parallelism": f"dp{world} (batch shards; loss boundary: {a.boundary})",
           "cache": f"inputs per step {a.batch * n_pts * FIN * 4 / 1e6:.0f} MB + weight-constant edge tables stream through HBM each step (> 126 MB L2); no explicit flush"}  # fmt: skip

    if a.impl == "reference":
        if rank != 0:
            return
        cfg["workload"] = f"{a.grid}_grid_{n_pts}pts_102to78_batch{a.batch}_per_gpu_f32"
        if a.grid != "1deg":
            emit({"impl": "reference", "unavailable": "the reference's replicated-graph decoder materialises ~22 GB fp32 per sample at 0.25 deg (BASELINE.md section 3): not run on CPU"})
            return
        # one step = one full forward at the step's batch (measured, not extrapolated); as many steps as fit ~4 minutes
        r = time_cpu_forward(lat_lons, a.batch, a.batch, max(1, a.steps), max(0, min(a.warmup, 1)), budget_s=200.0)
        sample = (f"full {a.batch}-sample forward per timed step on the 1deg grid; {r['steps']} timed + {r['warmup']} warm-up forwards actually ran "
                  f"(requested --steps {a.steps} --warmup {a.warmup}, cut to fit ~4 minutes)")  # fmt: skip
        emit({
            "impl": "reference", "metric": "forward steps/sec", "value": r["steps_per_s"], "unit": "steps/s", "n_gpus": a.gpus, "steps": r["steps"],
            "warmup": r["warmup"], "ms_per_step": 1000.0 / r["steps_per_s"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": r["steps_per_s"], "unit": "steps/s", "cores": r["cores"], "kind": r["kind"], "sample": sample},
            "e2e": {"value": r["steps_per_s"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        })  # fmt: skip
        return

    import __graft_entry__ as ge

    if rank == 0 or not os.path.exists(ge.LIB):
        ge.build()
    from graph_weather_b200 import GraphWeatherForecaster, NormalizedMSELoss, _capi
    from graph_weather_b200.dist import BoundaryGather

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_to_gpu_numa(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(42)
    # the drop-in call of the reference's README (README.md:52): no extra keyword on the default path
    model = (GraphWeatherForecaster(lat_lons) if a.precision == "auto" else GraphWeatherForecaster(lat_lons, precision=a.precision)).to(dev).eval()
    n, ed = n_pts, int(model.decoder._g_dec.src.size)
    torch.manual_seed(1234 + rank)
    x_host = torch.randn(a.batch, n, FIN).pin_memory()
    x = x_host.to(dev)
    out_host = torch.empty(a.batch, n, FOUT).pin_memory()
    gather = BoundaryGather(world * a.batch, dev, mode=a.gather_mode) if (world > 1 and a.boundary != "loss") else None
    crit = target = None
    if world > 1 and a.boundary == "loss":
        crit = NormalizedMSELoss([1.0] * FOUT, [tuple(p) for p in np.asarray(lat_lons).tolist()], normalize=False)
        target = torch.zeros(a.batch, n, FOUT, device=dev)

    def boundary(y):
        if world == 1:
            return y
        if crit is not None:
            return crit(y, target, total_batch=world * a.batch)  # one all-reduced scalar
        return gather(y, overlap=(a.boundary == "gather"))

    def forward_boundary(inp):
        """One step: the forward and whatever crosses GPUs at the loss boundary.  With the gather boundary the transfer is
        part of the forward's last kernel (BoundaryGather mode "fused") wherever symmetric memory is available."""
        if gather is not None:
            return gather.forward(model, inp, overlap=(a.boundary == "gather"))
        return boundary(model(inp))

    def step_resident():
        return forward_boundary(x)

    # End-to-end step through the public module call: every step copies its inputs in from pinned host memory and its
    # forecast back out.  The copies run on their own streams (double-buffered), so step i+1's input upload and step
    # i-1's download overlap step i's compute -- the steady state of a real rollout / evaluation loop.
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    x_bufs = [torch.empty_like(x), torch.empty_like(x)]
    out_bufs = [out_host, torch.empty_like(out_host).pin_memory()]
    e2e_state = {"i": 0, "used": [None, None], "dl": [None, None]}

    def step_e2e():
        i = e2e_state["i"]
        e2e_state["i"] = i + 1
        cur = torch.cuda.current_stream(dev)
        b = i & 1
        if e2e_state["used"][b] is not None:
            s_in.wait_event(e2e_state["used"][b])  # step i-2 has finished reading this input buffer
        with torch.cuda.stream(s_in):
            x_bufs[b].copy_(x_host, non_blocking=True)
            ev_in = torch.cuda.Event()
            ev_in.record(s_in)
        cur.wait_event(ev_in)
        if gather is not None:  # the gather buffer about to be written was downloaded two steps ago: that copy must be done
            kb = gather._i & 1
            if e2e_state["dl"][kb] is not None:
                cur.wait_event(e2e_state["dl"][kb])
        y = forward_boundary(x_bufs[b])
        if gather is not None:  # this rank's own rows of the gathered forecast are what it downloads
            y = y[rank * a.batch : (rank + 1) * a.batch]
        ev_c = torch.cuda.Event()
        ev_c.record(cur)
        e2e_state["used"][b] = ev_c
        s_out.wait_event(ev_c)
        with torch.cuda.stream(s_out):
            out_bufs[b].copy_(y, non_blocking=True)
            if gather is not None:
                ev_d = torch.cuda.Event()
                ev_d.record(s_out)
                e2e_state["dl"][kb] = ev_d
        y.record_stream(s_out)
        return y

    def sync_all():
        if gather is not None:
            gather.wait()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        cur = torch.cuda.current_stream(dev)
        if gather is not None:
            gather.wait()  # the timed region ends when the last gather has landed ...
        cur.wait_stream(s_in), cur.wait_stream(s_out)  # ... and the last download too
        e1.record()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)  # max over ranks
        sync_all()
        return float(ms.item()), out

    warm = max(3, a.warmup)
    for _ in range(warm):
        step_resident()
    plan = model._engine.plan
    plan.timing_enable(True)
    _capi.launch_count_reset()
    with ClockSampler(local) as clk:
        ms_total, y_last = timed(step_resident, a.steps)
    # copied now: the end-to-end steps below reuse the gather buffers
    dump = output_sample(y_last) if (a.dump_outputs and rank == 0) else None
    launches = _capi.launch_count()
    tags = plan.timing_read()
    plan.timing_enable(False)
    plan.status()  # raises if any kernel flagged fp16-range overflow or a pipeline fault
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, a.steps)
    ms_step = ms_total / a.steps
    value = world * a.steps / (ms_total / 1000.0)
    e2e_value = world * a.steps / (ms_e2e / 1000.0)
    resolved = model._engine.resolved_precision
    dtype = {"fp32": "f32 (fp16x2-split tcgen05, fp32 accumulate)", "fp32_tc": "f32 (fp16x2-split tcgen05, fp32 accumulate)",
             "fp32_simt": "f32", "bf16": "bf16"}[resolved]  # fmt: skip
    cfg["workload"] = f"{a.grid}_grid_{n_pts}pts_102to78_batch{a.batch}_per_gpu_{'bf16' if resolved == 'bf16' else 'fp32'}"
    cfg["precision"] = {"requested": a.precision, "resolved": resolved}
    cfg["plan_gib"] = round(plan.device_bytes() / 2**30, 2)
    if gather is not None:
        cfg["boundary_transport"] = {"mode": gather.mode, "fused_store": (gather._fused[0][0] if getattr(gather, "_fused", None) else None),
                                     "fallback_reason": gather.fallback_reason}  # fused_store 1 = NVLink multicast, 2 = peer stores

    # parity of THIS run: one sample of the bench's own batch against the CPU oracle (1 deg; checker only, outside any timing)
    parity = None
    if rank == 0 and not a.no_check:
        if a.grid == "1deg":
            from oracle import restate

            b = a.batch - 1
            with torch.no_grad():
                y = model(x)[b : b + 1].cpu()
            sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
            ref = restate.forecaster_forward(sd, oracle_graphs(model), x_host[b : b + 1])
            tol = 1e-4 if resolved != "bf16" else 2e-2
            err = float((y - ref).abs().max())
            parity = {"max_abs_err": err, "tol": tol, "ok": bool(err < tol), "sample": b, "oracle": "oracle/restate.py (CPU restatement pinned to the reference fixtures)"}
        else:
            parity = {"max_abs_err": None, "note": "no CPU oracle at 0.25 deg (22 GB/sample); see tests/test_gpu_parity.py::test_quarter_degree_*"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernels timed inside a seconds-long step loop)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    f_alg, per = algorithmic_flops(n, ed)
    dom = max((k for k in tags if tags[k][0] and k != "const"), key=lambda k: tags[k][1])
    cnt, ms_dom = tags[dom]
    per_launch_flops = per[dom] * a.batch * a.steps / cnt
    achieved = per_launch_flops / ((ms_dom / cnt) * 1e-3) / 1e12
    traffic, traffic_note = None, "no ncu capture of this build (profiles/traffic.json absent or measured on other sources)"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("source_hash") == source_hash() and tj.get("workload") == cfg["workload"]:
            traffic, traffic_note = tj.get(dom), "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, profiles/traffic.json (same sources, same workload)"
    except Exception:
        pass
    split_note = ("the fp32-faithful path issues 3 fp16 MMAs per product, so frac <= 1/3 x (algorithmic/executed FLOP ratio 1/0.58) = 0.57 of the bf16 peak"
                  if resolved in ("fp32", "fp32_tc") else "")  # fmt: skip
    roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                "note": "achieved = algorithmic (unfactored, SURVEY 8(d)) FLOPs per launch / mean launch time; " + split_note,
                "whole_step": {"achieved": f_alg * a.batch / (ms_step * 1e-3) / 1e12, "unit": "TFLOP/s",
                               "frac": f_alg * a.batch / (ms_step * 1e-3) / 1e12 / peak_tf},
                "per_kernel_ms_per_step": {k: round(v[1] / a.steps, 4) for k, v in tags.items() if v[0]},
                "kernel_time_share_of_step": round(sum(v[1] for v in tags.values()) / ms_total, 4)}  # fmt: skip
    line = {
        "metric": "forward steps/sec", "value": value, "unit": "steps/s", "n_gpus": world, "steps": a.steps, "warmup": warm,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype,
        "data": "synthetic", "config": cfg, "samples_per_s": value * a.batch,
        "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": int(out_host.numel() * 4),
                "ms_per_step": ms_e2e / a.steps, "numa_bound_cpus": numa_cpus},
        "gpu_launches": int(launches), "clocks": clk.summary(), "roofline": roofline, "parity": parity,
    }  # fmt: skip
    if world == 1 and not a.no_cpu_baseline and a.grid == "1deg":
        sample_b = min(2, a.batch)
        r = time_cpu_forward(lat_lons, a.batch, sample_b, 2, 1, budget_s=40.0)
        line["cpu_baseline"] = {"value": r["steps_per_s"], "unit": "steps/s", "cores": r["cores"], "kind": r["kind"], "seconds_per_forward": r["seconds_per_forward"],
                                "sample": f"reference forward on {sample_b} of the {a.batch} samples per timed forward ({r['warmup']} warm-up + {r['steps']} timed); steps/s = samples/s / {a.batch}; "
                                          "`bench.py --impl reference` times the full batch"}  # fmt: skip
    if dump is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    with torch.no_grad():  # an inference benchmark (forward steps/s): autograd off, like any evaluation loop
        main()
