#!/usr/bin/env python
"""bench.py -- throughput of the DSRG pixel-labelling hot path (BASELINE.json metric:
images/s for the SRG + DenseCRF pass at 321x321x21).

One "step" = one pass of the hot path over one batch of synthetic images:
  dsrg321 (default): DSRGLayer.forward body = dense-CRF refinement (10 mean-field iterations,
                     bilateral 80/13 + spatial 3, unary = probs) -> float64 clamp/renormalise ->
                     seeded region growing (th 0.99/0.85), batch 64 @ 321x321x21
  crf321 / srg321  : the CRF-only / SRG-only configurations of BASELINE.json (batch 64)
  full513          : the same full pass + balanced seeding loss, batch 16 @ 513x513x21
  sweep4096        : BASELINE config 5 -- 4096 images @ 321x321x21, image i on rank floor(i*R/4096)
                     (dsrg_b200/shard.py), each rank works through its shard in batches of 64: STRONG scaling.
                     The default (dsrg321) line also carries a `sweep4096` object measured in the same run.

`python bench.py --gpus N --steps K --warmup W` prints ONE JSON line (rank 0); the headline and `e2e` numbers
each time exactly K steps.  Under torchrun (WORLD_SIZE > 1) every rank runs the same per-rank batch on its own
GPU (images shard with no data-path collective; weak scaling) and the time is the max over ranks.

`--dump-outputs DIR` also writes what the timed path computed in its last timed step (rank 0's buffers) as
DIR/<name>.npy.  The inputs are seeded, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the reference's CPU path instead (oracle port: oracle/crf_oracle.c +
oracle/srg_oracle.py:srg_faithful) on all host cores; this and the `cpu_baseline` leg are the only
places bench.py touches oracle/.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    #            H    W    B   what
    "train41": (41, 41, 20, "crf+srg"),     # the shape the reference actually trains on (scale_factor 12)
    "dsrg321": (321, 321, 64, "crf+srg"),
    "crf321": (321, 321, 64, "crf"),
    "srg321": (321, 321, 64, "srg"),
    "full513": (513, 513, 16, "crf+srg+loss"),
    "sweep4096": (321, 321, 64, "crf+srg"),   # 4096 images in all, sharded; 64 = the batch a rank processes at a time
}
SWEEP_IMAGES = 4096
M = 21
T_ITERS = 10
TH1, TH2 = 0.99, 0.85


def algorithmic_bytes_per_image(what, N):
    """SURVEY.md 8(d): compulsory dense-array traffic per image."""
    b_srg = 252 * N                          # probs + cues in, seeds out: 3 * 4*C*N
    b_crf = N * (3 + 8 * M + 12 * M * T_ITERS)
    b_loss = 2 * 4 * M * N
    return {"crf": b_crf, "srg": b_srg, "crf+srg": b_crf + b_srg, "crf+srg+loss": b_crf + b_srg + b_loss}[what]


def kernel_survey_bytes(tag, N, B):
    """SURVEY.md 8(d) bytes ONE launch accounts for: the CRF budget is N(3 + 8M + 12MT), i.e. 12*M*N per image and
    mean-field iteration (read U, read Q, write Q), and one tile-kernel launch is one iteration."""
    per = {"mf_tile": 12 * M * N, "srg_label": 8 * M * N, "srg_emit": 4 * M * N, "mf_init": 12 * M * N, "mf_export": 8 * M * N}
    return per.get(tag, 0) * B


def kernel_algorithmic_bytes(tag, N, B):
    """Bytes ONE launch of a kernel class must move given OUR design, for a batch of B images."""
    per = {
        "mf_tile": 4 * M * N,           # the fused slice+update+splat kernel streams U once; Q stays on chip
        "mf_init": 8 * M * N + 4 * M * N,
        "srg_label": 8 * M * N,         # probs + cues
        "srg_emit": 4 * M * N,          # seeds out
        "mf_export": 8 * M * N,
    }
    return per.get(tag, 0) * B


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(object):
    """nvidia-smi sampling while the GPU is under load (B200_PROFILING.md clocks line).  Started
    before the warm-up steps so that nvidia-smi's start-up latency does not eat a short timed region;
    mark() is called at the start of the timed region and only later samples are reported when
    there are any."""

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.t_mark = None
        q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def mark(self):
        import datetime
        self.t_mark = datetime.datetime.now()

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f")
                rows.append((ts, float(c[1]), float(c[2]), float(c[3]), [n for n, v in zip(names, c[5:9]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        os.unlink(self.f.name)
        timed = [r for r in rows if self.t_mark is not None and r[0] >= self.t_mark]
        use, where = (timed, "timed region") if len(timed) >= 2 else (rows, "warm-up + timed region")
        if use:
            reasons = sorted(set(x for r in use for x in r[4]))
            out = {"sm_mhz": float(np.median([r[1] for r in use])), "sm_max_mhz": float(max(r[2] for r in use)),
                   "power_w_max": float(max(r[3] for r in use)), "reasons": reasons, "samples": len(use),
                   "sampled_during": where}
        return out


IMAGE_VARIANT = "smooth"


def usable_cpus():
    """CPUs this process can really use: affinity mask, further limited by the cgroup CPU quota (the GPU
    boxes expose 128 logical CPUs with a 16-CPU quota; oversubscribing only adds context switches)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        pass
    return n


DUMP_MAX_ELEMENTS = 1 << 22   # per array: 16 MB of float32, so the at most three arrays of a workload stay under 64 MB


def dump_outputs(directory, arrays):
    """Write each device tensor of ``arrays`` as directory/<name>.npy in float32 (float64 stays float64).  An array
    of more than DUMP_MAX_ELEMENTS elements is written as a sample of its flattened elements: the sorted distinct
    positions of DUMP_MAX_ELEMENTS draws of RandomState(0), the same in every run for the same shape."""
    import torch
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            pos = np.unique(np.random.RandomState(0).randint(0, t.numel(), DUMP_MAX_ELEMENTS))
            t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def synth_batch(H, W, B, unique=8):
    from dsrg_b200 import synth
    return synth.make_batch(B, H, W, cues="cam", image=IMAGE_VARIANT, unique=unique)


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU path (oracle port) -- also the cpu_baseline leg
# --------------------------------------------------------------------------------------------
def _cpu_one(args):
    what, labels, probs, cues, image = args
    from oracle import crf_oracle, loss_oracle, srg_oracle
    probs = probs.copy()
    out = None
    if "crf" in what:
        # refinement() with the image already at map resolution: pylayers.py:310-331 minus the zoom
        probs[probs < crf_oracle.MIN_PROB] = crf_oracle.MIN_PROB
        unary = np.ascontiguousarray(np.transpose(probs, (1, 2, 0)))
        # the reference's own CRF sources (oracle/_ref/libdensecrf_ref.so, built once in the dev container and
        # shipped with the snapshot) when present; the C restatement is bit-identical to it and equally fast
        crf = crf_oracle.CRF_reference if crf_oracle.ref_crf_available() else crf_oracle.CRF
        q = crf(image, unary, maxiter=T_ITERS, scale_factor=1.0)
        out = crf_oracle.renormalise(np.transpose(q, (2, 0, 1)))   # pylayers.py:328-330
    if "srg" in what:
        src = out if out is not None else probs.astype(np.float64)
        out = srg_oracle.srg_faithful(labels, cues, src, TH1, TH2)
    if "loss" in what:
        loss_oracle.balanced_seed_loss(probs[None], out[None], np.float32)
    return float(np.sum(out))


def cpu_kind(what):
    """'reference' only when everything timed is the reference's own compiled code (CRF-only workloads with
    oracle/_ref present); the SRG half is always the loop-for-loop Python port."""
    from oracle import crf_oracle
    return "reference" if (what == "crf" and crf_oracle.ref_crf_available()) else "port"


def cpu_crf_note():
    from oracle import crf_oracle
    return ("CRF = the reference's own CRF/src/*.cpp compiled in place (oracle/_ref)" if crf_oracle.ref_crf_available()
            else "CRF = oracle/crf_oracle.c (restatement)") + ", SRG = loop-for-loop port of generate_seed_step + CC_labeling_8"


def cpu_images_per_second(what, batch, n_images, cores, pool=None):
    items = [(what, batch["labels"][i % len(batch["labels"])], batch["probs"][i % len(batch["probs"])],
              batch["cues"][i % len(batch["cues"])], batch["image"][i % len(batch["image"])]) for i in range(n_images)]
    t = time.perf_counter()
    if pool is None:
        for it in items:
            _cpu_one(it)
    else:
        pool.map(_cpu_one, items, chunksize=1)   # items are pickled to the workers like pylayers.py:341-342
    dt = time.perf_counter() - t
    return n_images / dt, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import crf_oracle
    crf_oracle.build()
    H, W, B, what = WORKLOADS[args.workload]
    cores = usable_cpus()
    cores = max(1, min(cores, 64))  # every host thread we may use, capped at the batch size (26 MB pickled per image)
    n = cores  # one image per core per step: a bounded sample of the batch-64 workload
    batch = synth_batch(H, W, min(n, 8), unique=8)
    import multiprocessing as mp
    # one long-lived Pool like DSRGLayer.setup creates (pylayers.py:292); every image of a step goes
    # to a worker (the reference runs its CRF loop serially in the parent -- this arm is the
    # friendlier "all host threads" variant the bench contract asks for)
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(args.warmup):
            cpu_images_per_second(what, batch, n, cores, pool)
        t = time.perf_counter()
        for _ in range(args.steps):
            cpu_images_per_second(what, batch, n, cores, pool)
        dt = time.perf_counter() - t
    value = n * args.steps / dt
    sample = "%d images/step (1 per host thread) of the %s workload, %d steps, multiprocessing.Pool(%d)" % (n, args.workload, args.steps, cores)
    emit(json.dumps({
        "impl": "reference", "metric": "images/s, SRG + DenseCRF pass at %dx%dx%d" % (H, W, M), "value": value,
        "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "what": what, "H": H, "W": W, "labels": M, "mean_field_iters": T_ITERS,
                   "images_per_step": n},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": cpu_kind(what), "sample": sample,
                         "code": cpu_crf_note()},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
def run_b200(args, rank, local_rank, world):
    import torch
    from dsrg_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible; the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    H, W, B, what = WORKLOADS[args.workload]
    if args.batch:
        B = args.batch
    N = H * W
    batch = synth_batch(H, W, B)
    dev = torch.device("cuda", local_rank)
    eng = api.Engine(B, H, W, M, device=local_rank)
    params = api.crf_params(12.0 if args.workload == "train41" else 1.0, 13, T_ITERS)
    d_labels = torch.from_numpy(batch["labels"]).to(dev)
    d_probs = torch.from_numpy(batch["probs"]).to(dev)
    d_cues = torch.from_numpy(batch["cues"]).to(dev)
    d_image = torch.from_numpy(batch["image"]).to(dev)
    d_seeds = torch.empty_like(d_probs)
    d_unary = d_probs.permute(0, 2, 3, 1).contiguous() if what == "crf" else None   # one-off layout prep, untimed
    d_q = torch.empty_like(d_unary) if what == "crf" else None
    d_terms = torch.zeros(2, device=dev)

    from dsrg_b200 import shard

    def shard_sizes():
        """BASELINE config 5: this rank's contiguous share of the 4096-image job, in batches of at most B."""
        lo, hi = shard.shard_range(SWEEP_IMAGES, rank, world)
        return [min(B, hi - b) for b in range(lo, hi, B)]

    sweep = args.workload == "sweep4096"
    sizes = shard_sizes() if sweep else [B]
    images_per_step = SWEEP_IMAGES if sweep else world * B      # whole job, all ranks

    def one(nb):
        if what == "crf":
            eng.crf_dev(d_unary[:nb], d_image[:nb], params, d_q[:nb])
        elif what == "srg":
            eng.srg_dev(d_labels[:nb], d_probs[:nb], d_cues[:nb], TH1, TH2, d_seeds[:nb])
        else:
            eng.dsrg_forward_dev(d_labels[:nb], d_probs[:nb], d_cues[:nb], d_image[:nb], params, TH1, TH2, d_seeds[:nb])
            if "loss" in what:
                eng.seedloss_forward_dev(d_probs[:nb], d_seeds[:nb], d_terms)
                if dist is not None:
                    dist.all_reduce(d_terms)   # the path's only collective: 2 floats

    def step():
        for nb in sizes:
            one(nb)

    # a real stream (not the legacy default stream): repeated passes are then replayed as CUDA graphs
    side = torch.cuda.Stream(device=dev)
    _plain_step = step

    def step():
        with torch.cuda.stream(side):
            _plain_step()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(side)   # events on the stream the kernels are launched on
        for _ in range(steps):
            fn()
        e1.record(side)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step()
    eng.take_launch_count()
    if sampler:
        torch.cuda.synchronize()
        sampler.mark()
    # exactly --steps timed steps, one block (barrier + synchronize on both sides, max over ranks)
    ms = timed(step, args.steps)
    clocks = sampler.stop() if sampler else None
    launches = eng.take_launch_count()
    value = images_per_step * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path holds after its last step (dsrg_forward_dev also clamps probs in place);
        # taken before the legs below reuse the buffers
        outs = {"crf": {"crf_marginals": d_q}, "srg": {"seeds": d_seeds}}.get(what, {"seeds": d_seeds, "probs": d_probs})
        if "loss" in what:
            outs["loss_terms"] = d_terms
        dump_outputs(args.dump_outputs, outs)

    # per-kernel durations by CUDA events on the launching stream, same K steps repeated
    eng.profile(True)
    ms_prof = timed(step, args.steps)
    prof = eng.profile_read()
    eng.profile(False)
    peak, peak_src = measured_peak()
    total_kernel_ms = sum(v[0] for v in prof.values())
    # one mean-field iteration is a PAIR of launches: k_mf_tile over the plain tiles and k_mf_tile_hy over the hybrid
    # ones (textured images; an empty list on smooth ones) -- the roofline is taken on the pair
    prof_r = dict(prof)
    if "mf_tile" in prof_r and "mf_tile_hybrid" in prof_r:
        prof_r["mf_tile"] = (prof_r["mf_tile"][0] + prof_r.pop("mf_tile_hybrid")[0], prof_r["mf_tile"][1])
    top = max(prof_r.items(), key=lambda kv: kv[1][0]) if prof_r else None
    roofline = None
    kernels = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps,
                   "share": v[0] / total_kernel_ms} for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    if top:
        tag, (tms, cnt) = top
        per_launch_s = tms * 1e-3 / cnt
        sb = kernel_survey_bytes(tag, N, B)          # SURVEY.md 8(d): what `achieved` / `frac` are computed on
        ab = kernel_algorithmic_bytes(tag, N, B)     # what this design has to move (U once; Q stays on chip)
        ach = sb / per_launch_s / 1e9 if sb else 0.0
        traffic = None   # dram__bytes_read+write per launch from the last committed ncu --set full capture
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(tag)
            if tj and B and args.workload == "dsrg321":
                traffic = tj["dram_bytes_per_launch"] * B / tj["batch"]
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": tag, "launch": ("k_mf_tile + k_mf_tile_hy of the same iteration"
                                                                if tag == "mf_tile" and "mf_tile_hybrid" in prof else tag),
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "peak_source": peak_src,
                    "bytes_basis": "SURVEY.md 8(d): 12*M*N per image and mean-field iteration for the tile kernel",
                    "survey_bytes_per_launch": sb, "algorithmic_bytes_per_launch": ab,
                    "frac_own_bytes": (ab / per_launch_s / 1e9 / peak) if ab else None,
                    "traffic_over_survey_bytes": (traffic / sb) if (traffic and sb) else None,
                    "traffic_over_own_bytes": (traffic / ab) if (traffic and ab) else None,
                    "avg_launch_ms": per_launch_s * 1e3, "share_of_step": tms / total_kernel_ms,
                    "step_algorithmic_GBs": algorithmic_bytes_per_image(what, N) * B * args.steps / (ms * 1e-3) / 1e9,
                    "step_frac": algorithmic_bytes_per_image(what, N) * B * args.steps / (ms * 1e-3) / 1e9 / peak,
                    "profiled_ms_per_step": ms_prof / args.steps}

    # end to end through the host-buffer C-ABI entry point (pinned host memory, copies inside)
    e2e = None
    if what in ("crf+srg", "crf+srg+loss", "srg", "crf") and not args.no_e2e:
        h_labels = api.pinned_empty(batch["labels"].shape, np.float32); h_labels[...] = batch["labels"]
        h_probs = api.pinned_empty(batch["probs"].shape, np.float32); h_probs[...] = batch["probs"]
        h_cues = api.pinned_empty(batch["cues"].shape, np.float32); h_cues[...] = batch["cues"]
        h_image = api.pinned_empty(batch["image"].shape, np.uint8); h_image[...] = batch["image"]
        h_seeds = api.pinned_empty(batch["probs"].shape, np.float32)
        if what == "crf":
            h_unary = api.pinned_empty((B, H, W, M), np.float32); h_unary[...] = np.transpose(batch["probs"], (0, 2, 3, 1))
            h_q = api.pinned_empty((B, H, W, M), np.float32)

            def host_one(nb):
                eng.crf_host(h_unary[:nb], h_image[:nb], params, out=h_q[:nb])
            h2d, d2h = h_unary.nbytes + h_image.nbytes, h_q.nbytes
        elif what == "srg":
            def host_one(nb):
                eng.srg_host(h_labels[:nb], h_probs[:nb], h_cues[:nb], TH1, TH2, seeds_out=h_seeds[:nb])
            h2d, d2h = h_labels.nbytes + h_probs.nbytes + h_cues.nbytes, h_seeds.nbytes
        else:
            def host_one(nb):
                eng.dsrg_forward_host(h_labels[:nb], h_probs[:nb], h_cues[:nb], h_image[:nb], params, TH1, TH2,
                                      seeds_out=h_seeds[:nb])
            h2d = h_labels.nbytes + h_probs.nbytes + h_cues.nbytes + h_image.nbytes
            d2h = h_seeds.nbytes + h_probs.nbytes   # seeds + the in-place-clamped probs blob (travels as a bit mask)
        per_image_h2d, per_image_d2h = h2d / B, d2h / B

        def host_step():
            for nb in sizes:
                host_one(nb)
        h2d, d2h = per_image_h2d * sum(sizes), per_image_d2h * sum(sizes)
        for _ in range(1 if sweep else 2):
            host_step()
        def host_block():
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                host_step()          # synchronises its own stream before returning
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if dist is not None:
                t = torch.tensor([dt], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return dt
        dt = host_block()
        e2e = {"value": images_per_step * args.steps / dt, "unit": "images/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "api": "dsrg_*_host (C ABI, pinned host buffers)",
               "note": "inputs are re-sent from the same pinned buffers every step; the in-place 1e-4 clamp of probs "
                       "(pylayers.py:312) therefore only changes values during the first warm-up step"}

    extras = {}
    if args.workload == "dsrg321" and not args.no_extras and not args.no_e2e:
        # --- BASELINE config 5 in the same run: the 4096-image job sharded over the ranks (strong scaling) ---
        sw_sizes = shard_sizes()

        def sweep_dev():
            with torch.cuda.stream(side):
                for nb in sw_sizes:
                    one(nb)
        sw_ms = timed(sweep_dev, 1)
        barrier()
        t0 = time.perf_counter()
        for nb in sw_sizes:
            host_one(nb)
        torch.cuda.synchronize()
        sw_dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([sw_dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sw_dt = float(t.item())
        extras["sweep4096"] = {"what": "BASELINE config 5: %d images @ 321x321x21, contiguous shards (dsrg_b200/shard.py), "
                                       "batches of %d per rank" % (SWEEP_IMAGES, B),
                               "scaling": "strong", "images": SWEEP_IMAGES, "images_this_rank": int(sum(sw_sizes)),
                               "value": SWEEP_IMAGES / (sw_ms * 1e-3), "unit": "images/s", "ms": sw_ms,
                               "e2e": {"value": SWEEP_IMAGES / sw_dt, "unit": "images/s"}}
    if args.workload in ("dsrg321", "train41") and rank == 0 and world == 1 and not args.no_extras and not args.no_e2e:
        # --- through the plugin call itself: pylayers.DSRGLayer.forward on Caffe-style host blobs ---
        from dsrg_b200.dropin import caffe_shim
        caffe_shim.install()
        import pylayers
        sf = 12.0 if args.workload == "train41" else 1.0
        Hi = 321                                     # the net's input images are 321x321 whatever the map size
        if H == Hi:
            img = batch["image"]
        else:
            from dsrg_b200 import synth
            uniq = [synth.make_image(np.random.RandomState(50 + i), Hi, Hi, IMAGE_VARIANT) for i in range(min(B, 8))]
            img = np.stack([uniq[i % len(uniq)] for i in range(B)])
        net_images = np.ascontiguousarray(np.transpose(img.astype(np.float32) - np.array([104.0, 117.0, 123.0], np.float32),
                                                       (0, 3, 1, 2)))
        layer = pylayers.DSRGLayer()
        layer.param_str = "{'th1': %g, 'th2': %g, 'scale_factor': %g}" % (TH1, TH2, sf)
        bottom = [caffe_shim.Blob(batch["labels"].reshape(B, 1, 1, M)), caffe_shim.Blob(batch["probs"]),
                  caffe_shim.Blob(batch["cues"]), caffe_shim.Blob(net_images)]
        top = [caffe_shim.Blob()]
        layer.setup(bottom, top)
        layer.reshape(bottom, top)
        for _ in range(2):
            layer.forward(bottom, top)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            layer.forward(bottom, top)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        extras["e2e_layer"] = {"value": B * args.steps / dt, "unit": "images/s", "ms_per_step": 1e3 * dt / args.steps,
                               "api": "pylayers.DSRGLayer.forward (drop-in Python layer) on pageable numpy blobs of a "
                                      "pycaffe stand-in; the layer page-locks them on first use (cudaHostRegister), "
                                      "the float32 net images (B,3,%d,%d) are zoomed / mean-shifted / rounded on the "
                                      "device every step" % (Hi, Hi),
                               "h2d_bytes_per_step": int(sum(b.data.nbytes for b in bottom)),
                               "d2h_bytes_per_step": int(top[0].data.nbytes + bottom[1].data.nbytes)}
    if args.workload == "dsrg321" and not args.no_extras and not sweep:
        # --- the other image statistics: a 1/f "photo-like" spectrum and uniform noise (worst case) ---
        variants = {IMAGE_VARIANT: {"value": value, "ms_per_step": ms / args.steps}}
        for var in ("smooth", "photo", "noise"):
            if var in variants:
                continue
            from dsrg_b200 import synth
            uniq = [synth.make_image(np.random.RandomState(1234 + i), H, W, var) for i in range(min(B, 8))]
            imgs = np.stack([uniq[i % len(uniq)] for i in range(B)])
            d_image.copy_(torch.from_numpy(imgs).to(dev))
            for _ in range(3):
                step()
            vms = timed(step, 3)
            variants[var] = {"value": world * B * 3 / (vms * 1e-3), "ms_per_step": vms / 3}
        d_image.copy_(torch.from_numpy(batch["image"]).to(dev))
        extras["image_variants"] = {"unit": "images/s", "what": "device-resident, same probs / cues, image statistics varied: "
                                    "smooth = Gaussian-filtered noise, photo = 1/f amplitude spectrum, noise = uniform",
                                    "values": variants}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import crf_oracle
        crf_oracle.build()
        n = 6
        v, dt = cpu_images_per_second(what, batch, n, 1, None)
        cpu_baseline = {"value": v, "unit": "images/s", "cores": 1, "kind": cpu_kind(what), "code": cpu_crf_note(),
                        "sample": "%d images of the same %s batch, single thread like the reference's serial CRF loop "
                                  "(pylayers.py:325-326); %.1f s of CPU work" % (n, args.workload, dt)}
    if rank == 0:
        emit(json.dumps({
            "metric": "images/s, SRG + DenseCRF pass at %dx%dx%d" % (H, W, M), "value": value, "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if sweep else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": args.workload, "what": what, "H": H, "W": W, "labels": M, "batch_per_gpu": B,
                       "global_batch": SWEEP_IMAGES if sweep else B * world, "mean_field_iters": T_ITERS, "sigma": "bilateral 80/13, spatial 3, scale_factor %g" % (12.0 if args.workload == "train41" else 1.0),
                       "thresholds": [TH1, TH2], "images": "%s, cam-like cues, 8 distinct images repeated" % IMAGE_VARIANT,
                       "l2": "inputs larger than L2 (%.0f MB of probs+cues per step)" % (2 * 4 * M * N * B / 1e6),
                       "parallelism": "dp%d (images shard, no data-path collective)" % world},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "kernels": kernels, "cpu_baseline": cpu_baseline, **extras,
        }))
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


_JSON_OUT = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON result.  Libraries print there too (NCCL's version banner
    ignores NCCL_DEBUG_FILE at NCCL_DEBUG=VERSION), so fd 1 is pointed at stderr for the rest of the run
    and the JSON line is written to the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dsrg321", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="tuning aid: skip the host-buffer leg (the line is then not a valid result)")
    ap.add_argument("--no-extras", action="store_true", help="skip sweep4096 / e2e_layer / image_variants of the default line")
    ap.add_argument("--images", default="smooth", choices=["smooth", "photo", "noise"],
                    help="synthetic image variant: smooth (headline), photo (1/f spectrum) or uniform noise (worst "
                         "case: every tile overflows the shared-memory path)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (a fixed sample of large arrays, "
                         "64 MB at most)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    global IMAGE_VARIANT
    IMAGE_VARIANT = args.images
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
