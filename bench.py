#!/usr/bin/env python
"""Benchmark of the hot path: ray-samples/s on BASELINE.json's configs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--pass step|forward] [--config c2|c3|c4|c5] [--with-eikonal]
                  [--precision fp16x3|fp16|bf16] [--dump-outputs DIR]

Default = configs[1] (C2): fg-bob deformable field, 2048 rays x 128 samples per GPU, synthetic rays and synthetic
"trained-like" weights, ONE TRAINING STEP of the renderer per "step":
    weight packing (forward + transposed operands; weights change every optimiser step),
    training forward (fused query_field kernel writing the tape), compositing (render_pixel),
    loss = fixed linear functional of the rendered pixels, compositing backward, field backward (data-gradient kernel +
    weight-gradient kernel + per-frame chain), flat gradient buffer, and for N > 1 ONE NCCL all-reduce (mean) of it.
Rays shard data-parallel over the N GPUs (weak scaling: every rank renders its own batch).  `--pass forward` is the
inference path (query_field + render_pixel, no tape).  `value` times the step with inputs resident in HBM; `e2e` goes
through the same public API with the step's inputs in pinned HOST memory (H2D of rays + per-frame tables and D2H of the
rendered RGB inside the timed region).  `--config c4` is the strong-scaling shape of configs[3]: 4096 rays x (128 fg +
128 bg) samples, composed by depth, split over the ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

# algorithmic FLOPs per ray-sample (SURVEY.md 8d, hook-measured on the reference): F_query,fwd incl. the 1/16-ray
# eikonal forward (71 616 for fg fields), which this renderer does not compute.  Training step = 3 x forward (dgrad + wgrad).
FLOP_FWD = {"fg_bob": 1_914_380 - 71_616, "fg_skelhuman": 1_903_572 - 71_616, "comp": 1_479_732 - 35_808,
            # skel-human + DenseWarp (C5): the skel-human figure plus three soft-deformation stages of 2 x (199 x 256 + 256 x 256 + 3 x 256) FLOP
            "fg_comphuman": 1_903_572 - 71_616 + 3 * 2 * (199 * 256 + 256 * 256 + 3 * 256)}
CONFIGS = {
    "c2": dict(field="fg_bob", M=128, N=16, D=128, precision="fp16x3", desc="fg-bob 2048 rays x 128 samples per GPU (configs[1])"),
    "c3": dict(field="fg_skelhuman", M=256, N=16, D=192, precision="bf16", desc="skel-human 4096 rays x 192 samples per GPU, bf16 operands (configs[2])"),
    "c4": dict(field="comp", M=256, N=16, D=128, precision="fp16x3", desc="comp skel-quad+dense fg + bg, 4096 rays x 256 samples TOTAL, ray-sharded (configs[3])"),
    "c5": dict(field="fg_comphuman", M=256, N=16, D=128, precision="fp16x3", n_inst=50,
               desc="comp_skel-human_dense fg, 50 instance codes (frame f uses video f % 50), 4096 rays x 128 samples per GPU (configs[4])"),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), float(d["hbm_gbs"]), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


def dram_traffic_from_profile(kernel):
    """dram read+write bytes per launch of `kernel` from the committed ncu raw page (profiles/r02_*_raw.csv), else None."""
    import csv
    import glob

    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r02_*raw*.csv")), reverse=True):
        try:
            rows = list(csv.reader(open(path)))
            head = rows[0]
            ik, ir, iw = head.index("Kernel Name"), head.index("dram__bytes_read.sum"), head.index("dram__bytes_write.sum")
            units = rows[1]
            mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            vals = [float(r[ir].replace(",", "")) * mult.get(units[ir], 1.0) + float(r[iw].replace(",", "")) * mult.get(units[iw], 1.0)
                    for r in rows[2:] if kernel in r[ik]]
            if vals:
                return float(np.mean(vals)), os.path.basename(path)
        except Exception:
            continue
    return None, None


def kernel_shares_from_profile(precision):
    """Mean device time (us) of every product kernel of one training step from the committed ncu launch list
    (profiles/r02_launches_step_<precision>.csv; cold-cache, serialised: only the SHARES are used)."""
    import collections
    import csv

    for name in (f"r02_launches_step_{precision}.csv", "r02_launches_step_fp16.csv"):
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        rows = list(csv.reader(open(path)))
        hi = [i for i, r in enumerate(rows) if "Kernel Name" in r]
        if not hi:
            continue
        h = rows[hi[0]]
        ik, iv, iu = h.index("Kernel Name"), h.index("Metric Value"), h.index("Metric Unit")
        agg = collections.defaultdict(list)
        for r in rows[hi[0] + 1:]:
            if len(r) > iv:
                v = float(r[iv].replace(",", "")) * {"ns": 1e-3, "us": 1.0, "ms": 1e3}.get(r[iu], 1.0)
                agg[r[ik].split("(")[0].split("<")[0].split("::")[-1].replace("void ", "").strip()].append(v)
        # a kernel name can cover small side launches too (the eikonal instantiations of field_bwd_kernel / their wgrad jobs):
        # the step's main launch of a name is the cluster near its maximum
        return {k: float(np.mean([x for x in v if x >= 0.2 * max(v)])) for k, v in agg.items()}, name
    return None, None


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region, one nvidia-smi query loop (-lms) for the whole region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
        except Exception:
            pass

    def stop(self):
        time.sleep(0.25)  # let at least two samples land even for a short region
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=5)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def field_cfgs(name):
    from lab4d_b200 import spec

    return {"fg_bob": [spec.FG_BOB], "fg_skelhuman": [spec.FG_SKEL_HUMAN], "comp": [spec.BG, spec.FG_COMP_QUAD],
            "fg_comphuman": [spec.FieldConfig(motion="skel", B=18, symm_idx=spec.HUMAN_SYMM, dense=True)]}[name]


def make_problem(device, rank, field, M, N, D, n_inst=1):
    """Per field: (cfg, params, rays, tables); synthetic 'trained-like' weights, seeded rays.  n_inst > 1: every frame takes
    the instance code rows of video f % n_inst (RAC-style multi-video batches, lab4d/nnutils/embedding.py:259-281)."""
    import synth
    from lab4d_b200 import spec
    from test_gpu_parity import synth_tables

    out = []
    rays_np = synth.synth_rays(M, N, seed=10 + rank)
    for cfg in field_cfgs(field):
        st = synth.synth_state(spec.field_param_shapes(cfg), 0, cfg.category)
        P = {k: torch.from_numpy(v).to(device) for k, v in st.items()}
        rays = {k: torch.from_numpy(v).to(device) for k, v in rays_np.items()}
        if cfg.category == "bg" and field == "comp":
            rays["near_far"] = rays["near_far"] * torch.tensor([[0.93, 1.11]], device=device)
        tab = {k: v.clone() for k, v in synth_tables(cfg, M, device, seed=10 + rank, rays=rays, P=P).items()}
        if n_inst > 1:
            g = torch.Generator().manual_seed(77)
            vid = torch.arange(M) % n_inst
            for k in [k for k in tab if k.startswith("inst_")]:
                tab[k] = (0.5 * torch.randn(n_inst, tab[k].shape[-1], generator=g))[vid].to(device).contiguous()
        out.append((cfg, P, rays, tab))
    return out


def dump_outputs(path, rend, renderers, train, limit=64 << 20):
    """Write what one step of the timed path hands its caller - the rendered pixels and, for a training step, every hot-path
    parameter's gradient (per field) - as float32 DIR/<name>.npy.  An array larger than its equal share of `limit` bytes is
    replaced by a fixed sample of its flattened elements (seeded by the array's size, so two runs pick the same ones)."""
    arrs = {f"rend.{k}": v for k, v in sorted(rend.items())}
    if train:
        for fi, r in enumerate(renderers):
            arrs.update({f"grad.{fi}.{k}": v for k, v in r.grad_buffer()[1].items()})
    share = limit // (4 * len(arrs))
    os.makedirs(path, exist_ok=True)
    for name, t in arrs.items():
        a = t.detach().float().cpu()
        if a.numel() > share:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(a.numel()))[:share].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a.numpy())


# ------------------------------------------------------------------------------------------ CPU arm (reference's PyTorch path)
def cpu_reference_rate(field, M, N, D, with_backward, reps, threads):
    """The reference's CPU PyTorch implementation of the path on the host cores: the UNMODIFIED reference (oracle/_ref
    through oracle/ref_shims) when that copy is present, else the oracle port."""
    torch.set_num_threads(threads)
    kind = "port"
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_shims"))
        import _install

        if not _install.available() or field != "fg_bob":
            raise ImportError
        import ref_harness as H
        import synth
        from lab4d.utils.render_utils import render_pixel as ref_render_pixel

        mf = H.build_field("fg", "bob", seed=0)
        fld = mf.field_params["fg"]
        H.set_n_depth(D)
        Kinv, batch = H.make_batch(fld, synth.synth_rays(M, N, seed=10))

        def step():
            fld.zero_grad()
            s = fld.get_samples(Kinv, batch)
            feat, deltas, _ = fld.query_field(s, flow_thresh=None)
            r = ref_render_pixel(feat, deltas)
            if with_backward:
                (r["rgb"].sum() + r["mask"].sum() + 1e-3 * r["flow"].sum()).backward()
        kind = "reference"
    except Exception:
        import lab4d_oracle as O

        cfg, P, rays, tab = make_problem("cpu", 0, field, M, N, D)[-1]
        if with_backward:
            P = {k: v.requires_grad_(True) for k, v in P.items()}

        def step():
            feat, deltas = O.query_field(P, cfg.as_oracle_cfg(), rays, tab, D)
            r = O.render_pixel(feat, deltas)
            if with_backward:
                for v in P.values():
                    v.grad = None
                (r["rgb"].sum() + r["mask"].sum() + 1e-3 * r["flow"].sum()).backward()
    ctx = torch.enable_grad() if with_backward else torch.no_grad()
    with ctx:
        step()
        t0 = time.perf_counter()
        for _ in range(reps):
            step()
        dt = (time.perf_counter() - t0) / reps
    return M * N * D / dt, dt, kind


def cpu_policy():
    """Fixed thread policy: all host cores (os.cpu_count()), capped at 32 - beyond that PyTorch's intra-op pool only adds
    contention for this op mix of hundreds of small kernels."""
    ncpu = os.cpu_count() or 1
    return min(ncpu, 32), ncpu


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation on the host cores (rank 0 only), bounded sample per step."""
    if rank != 0:
        return
    cfgd = CONFIGS[args.config]
    threads, ncpu = cpu_policy()
    Ms = 8
    with_bwd = args.passes == "step"
    times, kind = [], "port"
    for i in range(args.warmup + args.steps):
        rate, dt, kind = cpu_reference_rate(cfgd["field"] if cfgd["field"] != "comp" else "fg_bob", Ms, cfgd["N"], cfgd["D"], with_bwd, 1, threads)
        if i >= args.warmup:
            times.append(dt)
    S = Ms * cfgd["N"] * cfgd["D"]
    val = S / float(np.mean(times))
    sample = f"{Ms} of {cfgd['M']} frames x {cfgd['N']} rays x {cfgd['D']} samples per step, {'forward+backward' if with_bwd else 'forward'}, fp32"
    print(json.dumps({
        "impl": "reference", "metric": "ray-samples/s", "value": val, "unit": "ray-samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfgd["desc"] + (", training step" if with_bwd else ", forward"), "sample": sample, "pass": args.passes},
        "cpu_baseline": {"value": val, "unit": "ray-samples/s", "cores": threads, "host_cores": ncpu, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------ GPU arm
class Step:
    """One step of the chosen pass over one batch, through the public API (lab4d_b200.render / autograd / parallel)."""

    def __init__(self, args, device, rank, world):
        from lab4d_b200 import parallel
        from lab4d_b200.render import FieldRenderer

        cfgd = CONFIGS[args.config]
        self.cfgd, self.args, self.device, self.world = cfgd, args, device, world
        M = cfgd["M"]
        if args.config == "c4":  # strong scaling: the 4096 rays are split over the ranks (frame pairs stay together)
            lo, hi = parallel.shard_frames(M, rank, world)
            M = hi - lo
        self.M, self.N, self.D = M, cfgd["N"], cfgd["D"]
        self.S = self.M * self.N * self.D * len(field_cfgs(cfgd["field"]))
        self.fields = make_problem(device, rank, cfgd["field"], self.M, self.N, self.D, n_inst=cfgd.get("n_inst", 1))
        self.precision = args.precision or cfgd["precision"]
        self.renderers = [FieldRenderer(cfg, device, operand_dtype=self.precision) for cfg, *_ in self.fields]
        self.train = args.passes == "step"
        if self.train:
            for _, P, _, _ in self.fields:
                for v in P.values():
                    v.requires_grad_(True)
            g = torch.Generator().manual_seed(5)
            R = self.M * self.N
            self.coeff = {k: (torch.rand(self.M, self.N, c, generator=g) / R).to(device) for k, c in
                          (("rgb", 3), ("mask", 1), ("depth", 1), ("flow", 2), ("feature", 16), ("vis", 1), ("xyz", 3), ("gauss_mask", 1),
                           ("mask_fg", 1), ("cyc_dist", 1))}
        self.launches = 0
        self.flat = None
        self.ctxs = {}
        g = torch.Generator().manual_seed(6)
        self.eik_rays = torch.randperm(self.M * self.N, generator=g)[:max(self.M * self.N // 16, 1)].to(device=device, dtype=torch.int32)

    def run(self, fields=None):
        from lab4d_b200 import autograd as b2grad
        from lab4d_b200 import parallel
        from lab4d_b200.render import compose_fields, render_pixel

        fields = fields or self.fields
        feats, dls = [], []
        for r, (cfg, P, rays, tab) in zip(self.renderers, fields):
            if self.train:
                r.pack_train(P)
                feat, deltas, self.ctxs[id(r)] = b2grad.query_field(r, P, rays, tab, self.D, bind_grads=True, return_ctx=True)
                self.launches += 2 + 2  # pack, pack^T; prologue + field_fwd(train)
            else:
                r.pack(P)
                feat, deltas = r.query_field(P, rays, tab, self.D)
                self.launches += 1 + 2
            feats.append(feat)
            dls.append(deltas)
        if self.train and self.args.with_eikonal:  # NeRF.compute_eikonal on R/16 rays of every field (nnutils/nerf.py:416-453)
            for r, (cfg, P, rays, tab), feat in zip(self.renderers, fields, feats):
                g = b2grad.eikonal(r, self.ctxs[id(r)], P, self.eik_rays, bind_grads=True)
                eik = torch.zeros(self.M * self.N, self.D, device=self.device)
                eik[self.eik_rays] = (g.norm(2, dim=-1) - 1) ** 2
                feat["eikonal"] = eik.view(self.M, self.N, self.D, 1)
                self.launches += 1 + 1 + 4  # reverse chain; absmax, scale, chain A, chain B, weight gradients
        fd, dl = (feats[0], dls[0]) if len(feats) == 1 else compose_fields(feats, dls)
        rend = render_pixel(fd, dl)
        self.launches += 1 + (len(feats) > 1) * 2
        if self.train:
            loss = sum((self.coeff[k] * rend[k]).sum() for k in self.coeff if k in rend)
            if self.args.with_eikonal:
                loss = loss + 1e-3 * rend["eikonal"].mean()
            for _, P, _, _ in fields:
                for v in P.values():
                    v.grad = None
            loss.backward()
            self.launches += 1 + 6  # composite_bwd; prologue, absmax, scale, field_bwd, wgrad, chain
            # the parameters' .grad are views of the renderers' flat gradient buffers: the step's all-reduce runs on them
            # (one NCCL call per field: 1 for C2 / C3, 2 for the composed scene)
            self.flat = [r.grad_buffer()[0] for r in self.renderers]
            for fl in self.flat:
                parallel.allreduce_mean_(fl)
        return rend


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--pass", dest="passes", default="step", choices=["step", "forward"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--precision", default=None, choices=["fp16x3", "fp16", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--with-eikonal", action="store_true",
                    help="the step also evaluates the eikonal term on 1/16 of the rays (reverse chain, loss, forward chains + weight gradients: "
                         "NeRF.compute_eikonal and its second-order backward)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of replaying the step as a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's rendered outputs and parameter gradients to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch.distributed as dist

    from lab4d_b200.render import HostStage

    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    step = Step(args, device, rank, world)
    cfgd = step.cfgd
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)  # > 126 MB L2

    # end-to-end arm: the step's inputs (rays + per-frame tables of every field) live in ONE pinned host arena
    host = {}
    for fi, (_, _, rays, tab) in enumerate(step.fields):
        for k, v in {**rays, **tab}.items():
            host[f"{fi}/{k}"] = v.detach().cpu()
    stage = HostStage(host, device)
    rgb_host = torch.empty(step.M, step.N, 3).pin_memory()

    def step_e2e():
        dev = stage.upload()
        fields = []
        for fi, (cfg, P, rays, tab) in enumerate(step.fields):
            fields.append((cfg, P, {k: dev[f"{fi}/{k}"] for k in rays}, {k: dev[f"{fi}/{k}"] for k in tab}))
        rend = step.run(fields)
        rgb_host.copy_(rend["rgb"].detach(), non_blocking=True)
        return rend

    def timed(fn, steps):
        """Per-step times (ms) of `steps` calls of fn, and what the last call returned."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        out = None
        for i in range(steps):
            flush.fill_(i & 0xFF)  # evict L2 between timed iterations
            ev[i][0].record()
            out = fn()
            ev[i][1].record()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in ev], out

    for _ in range(args.warmup):
        step.run()
        step_e2e()
    torch.cuda.synchronize()
    # the step as one CUDA graph (static shapes): replaying keeps the host out of the timed region
    run_fn, e2e_fn, graphed = step.run, step_e2e, False
    if not args.no_graph:
        try:
            from lab4d_b200.graph import GraphedStep

            g_run = GraphedStep(step.run, warmup=2, device=device)
            g_e2e = GraphedStep(step_e2e, warmup=2, device=device)
            run_fn, e2e_fn, graphed = g_run.replay, g_e2e.replay, True
        except Exception as ex:  # stay on the eager path
            print(f"bench: CUDA-graph capture failed ({type(ex).__name__}: {str(ex)[:200]}); eager launches", file=sys.stderr)
            torch.cuda.synchronize()
    launches_per_step = None
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    step.launches = 0
    step.run()
    launches_per_step = step.launches
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    ms, last_rend = timed(run_fn, args.steps)
    n_launch = launches_per_step * args.steps
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:  # before the end-to-end arm's steps overwrite the gradient buffers
        dump_outputs(args.dump_outputs, last_rend, step.renderers, step.train)
    ms_e2e, _ = timed(e2e_fn, args.steps)
    # the phases alone: the forward call and the backward call of the (last) field, each replayed as its own CUDA graph and
    # timed with CUDA events on the launching stream
    phase = {"fwd_ms": [], "bwd_ms": []}
    r0, (cfg0, P0, rays0, tab0) = step.renderers[-1], step.fields[-1]
    P0d = {k: v.detach() for k, v in P0.items()}
    hold = {}

    def ph_fwd():
        if step.train:
            hold["feat"], _, hold["ctx"] = r0.query_field_train(P0d, rays0, tab0, step.D)
        else:
            hold["feat"], _ = r0.query_field(P0d, rays0, tab0, step.D)

    def ph_bwd():
        f = hold["feat"]
        r0.backward(hold["ctx"], {"rgb": f["rgb"], "density": f["density"], "vis": f["vis"], "xyz": f["xyz"]})

    try:
        from lab4d_b200.graph import GraphedStep

        if args.no_graph:
            raise RuntimeError("eager")
        gf = GraphedStep(ph_fwd, warmup=2, device=device)
        gb = GraphedStep(ph_bwd, warmup=2, device=device) if step.train else None
        f_fn, b_fn = gf.replay, (gb.replay if gb else None)
    except Exception:
        f_fn, b_fn = ph_fwd, (ph_bwd if step.train else None)
    # the eikonal term alone (R/16 rays): reverse chain, then forward chains + weight gradients, as their own graph
    eik_ms = []
    if step.train and not args.no_graph:
        try:
            ph_fwd()
            n_e = int(step.eik_rays.numel())
            gbar = (1e-6 * torch.randn(n_e, step.D, 3, generator=torch.Generator().manual_seed(8))).to(device)
            eflat = torch.zeros(r0._train_state()["total"], device=device)

            def ph_eik():
                _, ectx = r0.eikonal_forward(hold["ctx"], step.eik_rays)
                r0.eikonal_backward(hold["ctx"], ectx, gbar, flat=eflat)

            ge = GraphedStep(ph_eik, warmup=2, device=device)
            for i in range(20):
                flush.fill_(i & 0xFF)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ge.replay()
                e1.record()
                torch.cuda.synchronize()
                eik_ms.append(e0.elapsed_time(e1))
            ge = None
        except Exception as ex:
            print(f"bench: eikonal phase not timed ({type(ex).__name__}: {str(ex)[:160]})", file=sys.stderr)
    for i in range(min(args.steps, 50)):
        flush.fill_(i & 0xFF)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        f_fn()
        e[1].record()
        if b_fn:
            b_fn()
        e[2].record()
        torch.cuda.synchronize()
        phase["fwd_ms"].append(e[0].elapsed_time(e[1]))
        phase["bwd_ms"].append(e[1].elapsed_time(e[2]))
    # the inference path of the same batch (no tape), parity mode and fast mode: short graph replays, reported beside the step
    fwd_variants = {}
    if step.train and len(step.fields) == 1 and not args.no_graph:
        from lab4d_b200.render import FieldRenderer, render_pixel

        for prec in ("fp16x3", "fp16"):
            try:
                rf = FieldRenderer(cfg0, device, operand_dtype=prec)

                def fwd_only():
                    rf.pack(P0d)
                    ft, dl = rf.query_field(P0d, rays0, tab0, step.D)
                    return render_pixel(ft, dl)

                gfo = GraphedStep(fwd_only, warmup=2, device=device)
                tms, _ = timed(gfo.replay, 20)
                fwd_variants[prec] = {"ms_per_step": float(np.mean(tms)), "value_per_gpu": step.S / (float(np.mean(tms)) * 1e-3), "unit": "ray-samples/s",
                                      "what": "pack + query_field + render_pixel, no tape"}
                gfo = None
            except Exception as ex:
                fwd_variants[prec] = {"error": str(ex)[:120]}
    # the same step with the eikonal term inside (R/16 rays: reverse chain, loss, forward chains, weight gradients), beside the default
    step_variants = {}
    if step.train and not args.with_eikonal and not args.no_graph and len(step.fields) == 1 and world == 1:
        try:
            import copy

            a2 = copy.copy(args)
            a2.with_eikonal = True
            st2 = Step(a2, device, rank, world)
            for _ in range(3):
                st2.run()
            g2 = GraphedStep(st2.run, warmup=2, device=device)
            tms, _ = timed(g2.replay, 30)
            step_variants["with_eikonal"] = {"ms_per_step": float(np.mean(tms)), "value_per_gpu": st2.S / (float(np.mean(tms)) * 1e-3), "unit": "ray-samples/s",
                                             "what": "the default step + NeRF.compute_eikonal on 1/16 of the rays and its second-order backward (eikonal kernels)"}
            g2 = st2 = None
        except Exception as ex:
            step_variants["with_eikonal"] = {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}
    clocks = sampler.stop()
    tot = torch.tensor([sum(ms), sum(ms_e2e)], device=device, dtype=torch.float64)
    Stot = torch.tensor([float(step.S)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        dist.all_reduce(Stot, op=dist.ReduceOp.SUM)
    ms_step = float(tot[0]) / args.steps
    ms_step_e2e = float(tot[1]) / args.steps
    if rank == 0:
        peak_burst, peak_sust, peak_bw, how = peaks()
        S_all = float(Stot[0])
        flop_fwd = FLOP_FWD[cfgd["field"]]
        fwd_ms = float(np.mean(phase["fwd_ms"]))
        bwd_ms = float(np.mean(phase["bwd_ms"])) if step.train else 0.0
        mult = 3 if step.train else 1
        kern_ms = fwd_ms + bwd_ms
        achieved = mult * flop_fwd * step.S / (kern_ms * 1e-3) / 1e12 if len(step.fields) == 1 else None
        kname = "field_fwd_kernel"
        traffic, tsrc = dram_traffic_from_profile(kname)
        strong = args.config == "c4"
        line = {
            "metric": "ray-samples/s", "value": S_all / (ms_step * 1e-3), "unit": "ray-samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": {"fp16x3": "f16 head+tail operands (3 MMAs per k-step, ~fp32 results: meets the 1e-4 RGB contract) / f32 accumulate",
                      "fp16": "f16 operands / f32 accumulate", "bf16": "bf16 operands / f32 accumulate"}[step.precision]
                     + ("; backward GEMMs f16 (scaled) / f32 accumulate" if step.train else ""),
            "data": "synthetic",
            "config": {"workload": cfgd["desc"] + (", training step (fwd + bwd + grad all-reduce)" if step.train else ", forward query_field + render_pixel")
                                   + (" + eikonal term on 1/16 of the rays" if step.train and args.with_eikonal else ""),
                       "pass": args.passes, "precision": step.precision, "rays_per_gpu": step.M * step.N, "samples_per_ray": step.D * len(step.fields),
                       "l2": "flushed between iterations (256 MB write)", "per_gpu": "BASELINE metric ray-samples/s/GPU = value / n_gpus",
                       "parallelism": f"dp{world}: rays sharded" + (", one NCCL all-reduce (mean) of the flat gradient buffer per step" if step.train else ", no data-path collective in forward")},
            "e2e": {"value": S_all / (ms_step_e2e * 1e-3), "unit": "ray-samples/s", "h2d_bytes_per_step": stage.nbytes,
                    "d2h_bytes_per_step": rgb_host.numel() * 4},
            "gpu_launches": n_launch, "cuda_graph": graphed,
            "phases_ms": {"forward_call": fwd_ms, "backward_call": bwd_ms, "step": ms_step,
                          "eikonal_call": (float(np.mean(eik_ms)) if eik_ms else None),
                          "eikonal_note": "b200r_eikonal_fwd + b200r_eikonal_bwd on R/16 rays (reverse chain, 2 forward chains, weight gradients); "
                                          + ("inside the step" if args.with_eikonal else "NOT inside the step (--with-eikonal adds it)"),
                          "note": "CUDA events around FieldRenderer.query_field[_train] (prologue + field kernel) and FieldRenderer.backward (prologue, scale, data-gradient kernel, weight-gradient kernel, per-frame chain)"},
            "clocks": clocks, "wall_s_timed_region": t_wall,
        }
        if achieved is not None:
            line["roofline"] = {"bound": "tensor", "kernel": "field_fwd_kernel + field_bwd_kernel + wgrad_kernel" if step.train else "field_fwd_kernel",
                                "achieved": achieved, "peak": peak_burst, "unit": "TFLOP/s", "frac": achieved / peak_burst,
                                "frac_of_sustained": achieved / peak_sust, "traffic": traffic,
                                "traffic_unit": f"DRAM bytes per field_fwd launch ({tsrc})" if tsrc else "no committed ncu capture found",
                                "kernel_ms": kern_ms, "flop_per_sample": mult * flop_fwd,
                                "peak_source": how + " bf16 dense burst (sustained also given)"}
        if step.train and len(step.fields) == 1:
            # per-kernel view: the backward call's measured time is split by the committed launch list's shares; the tape
            # makes the two backward kernels HBM-bound by design (bytes = chunks each kernel must move, DESIGN.md 4)
            shares, src = kernel_shares_from_profile(step.precision)
            tiles = step.M * ((step.N * step.D + 127) // 128)
            chunks = {"fg_bob": (79, 82, 161), "fg_skelhuman": (76, 82, 158)}.get(cfgd["field"])
            if shares and chunks and "field_bwd_kernel" in shares and "wgrad_kernel" in shares:
                tb = shares["field_bwd_kernel"] + shares["wgrad_kernel"]
                bwd_k = {k: bwd_ms * shares[k] / tb for k in ("field_bwd_kernel", "wgrad_kernel")}
                rk = []
                a_b, g_b, u_b = (c * 16384.0 * tiles for c in chunks)
                for kname, ms_k, nbytes in (("field_fwd_kernel (training forward)", fwd_ms, a_b), ("field_bwd_kernel", bwd_k["field_bwd_kernel"], g_b),
                                            ("wgrad_kernel", bwd_k["wgrad_kernel"], u_b)):
                    gbs = nbytes / (ms_k * 1e-3) / 1e9
                    tr, _ = dram_traffic_from_profile(kname.split(" ")[0])
                    rk.append({"kernel": kname, "bound": "hbm", "ms": ms_k, "achieved": gbs, "peak": peak_bw, "unit": "GB/s", "frac": gbs / peak_bw,
                               "algorithmic_bytes": nbytes, "traffic": tr})
                line["roofline_kernels"] = {"kernels": rk, "split_source": f"profiles/{src} (shares of the backward call)",
                                            "note": "tape bytes each kernel must write / read once: forward 79, data-gradient 82, weight-gradient 161 chunks of 16 KB per 128-sample tile"}
        if fwd_variants:
            line["forward_only"] = fwd_variants
        if step_variants:
            line["step_variants"] = step_variants
        if step.flat is not None:
            line["grad_buffer_bytes"] = int(sum(fl.numel() for fl in step.flat) * 4)
        if not args.no_cpu_baseline and world == 1 and args.config == "c2":  # reported baseline: rank 0 at N = 1, ~10-20 s of CPU work
            threads, ncpu = cpu_policy()
            Ms, reps = 8, (12 if step.train else 40)
            rate, dt, kind = cpu_reference_rate(cfgd["field"], Ms, step.N, step.D, step.train, reps, threads)
            line["cpu_baseline"] = {"value": rate, "unit": "ray-samples/s", "cores": threads, "host_cores": ncpu, "kind": kind,
                                    "sample": f"{reps} x ({Ms} of {cfgd['M']} frames x {step.N} rays x {step.D} samples), "
                                              f"{'forward+backward' if step.train else 'forward'}, fp32, {reps * dt:.1f} s"}
        print(json.dumps(line), flush=True)
    # tear-down: graphs that captured NCCL collectives must go before the process group does; then an ordinary interpreter
    # exit (exit handlers and library destructors run)
    g_run = g_e2e = gf = gb = run_fn = e2e_fn = f_fn = b_fn = None
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
