"""Headline benchmark: federated rounds/second (BASELINE.json) — ResNet-18 / FedCIFAR-100 by default, ``--task`` for the
other BASELINE configs.

    python bench.py --gpus N --steps K --warmup W [--task T]      # this framework
    python bench.py --impl reference --gpus N ... [--task T]      # the unmodified reference from baseline/_ref

One "step" = one FL round of the benchmark config.  Flagship: 10 sampled clients x (100 samples, batch 20 => 5 local
SGD steps, clip 5.0, gradient statistics) + weighted aggregation + server SGD(lr 1.0) + model (re)distribution + the
per-round ``latest_model.tar`` checkpoint.  Synthetic data of the benchmark's shape, random-init weights.  For N > 1
launch under ``torch.distributed.run`` (one rank per GPU).

What is measured (all through the public API ``OptimizationServer.begin_training / run_rounds``):

* ``value``: K rounds bracketed by ``Server.sync_nodes()`` (every rank drains its GPU, records a CUDA event, barriers);
  each rank reports its own device time between its events, the maximum over ranks is used.  Before the W warm-up
  rounds the job runs set-up rounds until two consecutive rounds agree within 5 % (CUDA-graph capture, peer mappings,
  allocator growth happen there), so the timed window is steady state; ``median_ms_per_round`` (per-round CUDA events
  on rank 0, which waits for every peer inside the fused update) is reported next to it.
* ``exposed_comm``: device time per round of the model distribution + gradient gather phases (slot scatter-in, fused
  pseudo-gradient accumulation, cross-GPU reduce + server update + broadcast kernel incl. its barriers), max over
  ranks.  Everything of a round runs on one stream, so these are exposed (not overlapped with client compute); for
  N > 1 the NVLink roofline fraction is reported with it.
* ``e2e``: the K rounds again with the engines in streaming mode: every round's client shards are copied
  host(pinned)->device inside the timed region and the round's record table is read back; wall clock.
* ``--sync-ckpt`` writes ``latest_model.tar`` synchronously every round like the reference (default: async
  latest-wins writer); ``--norm bn`` runs the reference's as-shipped BatchNorm variant of the model.

``--dump-outputs DIR`` writes what the last timed round returned to its caller, for comparing two builds output for
output: ``train_loss.npy`` (float64, the loss ``run_rounds`` returned) and ``global_model.npy`` (float32, every
floating-point tensor of the updated global model's state dict, flattened in order; a model of more than
``DUMP_MAX_VALUES`` entries is written as a fixed, seeded sample of them).  Data, model init and client sampling are
seeded and the set-up phase runs a fixed ``SETUP_ROUNDS_FIXED`` rounds, so every round has the same index and client
sample on every run.  The last timed round also starts from the seeded initial global model, copied back in place
before it: float atomics reorder the gradient sums of every earlier round, and training (GroupNorm over 2-channel
groups on 1x1 maps) amplifies those last-bit differences round after round, so the weights it would otherwise start
from differ between runs.  The dumped round thus has the same inputs on every run.

``gpu_launches`` counts launches of this repo's own kernels in the timed region (rank 0).
``FLUTE_BENCH_CPU=1`` runs the same protocol on CPU/gloo with a tiny population (control-flow test, no number).
"""
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "baseline"))
from bench_common import (BASELINE_PUBLISHED, TASKS, ClockSampler, emit, parse_args)  # noqa: E402

SETUP_ROUNDS_FIXED = 8              # with --dump-outputs; _settle() usually stops after 4-5 rounds
DUMP_MAX_VALUES = 15_000_000        # float32 entries of global_model.npy: 60 MB, keeps a dump under 64 MB


def _reference(args):
    """Re-exec into a clean interpreter so nothing of this repo is importable on the reference's path."""
    os.environ["PYTHONPATH"] = ""
    script = os.path.join(ROOT, "baseline", "run_reference.py")
    os.execv(sys.executable, [sys.executable, script] + sys.argv[1:])


class BenchJob:
    def __init__(self, server, worker, comm, config):
        self.server, self.worker, self.comm, self.config = server, worker, comm, config
        self._begun = False

    def run_round(self):
        if not self._begun:
            self.server.begin_training()
            self._begun = True
        return self.server.run_rounds(1)

    def close(self):
        if self._begun:
            self.server.end_training()


FlagshipJob = BenchJob


def make_config(task="cv_resnet_fedcifar100", n_clients_per_round=None, rounds=10 ** 6, norm="gn", comm="auto",
                resident=True, compute_dtype=None, sync_ckpt=False):
    import yaml
    from msrflute_b200.core.config import FLUTEConfig
    spec = TASKS[task]
    with open(os.path.join(ROOT, "experiments", task, "config.yaml")) as f:
        raw = yaml.safe_load(f)
    sc = raw["server_config"]
    sc["max_iteration"] = rounds
    sc["num_clients_per_iteration"] = n_clients_per_round or spec["clients_per_round"]
    sc["val_freq"], sc["rec_freq"] = 10 ** 9, 10 ** 9      # rounds only (the reference arm does the same)
    sc["initial_val"], sc["initial_rec"] = False, False
    b200 = sc.setdefault("b200", {})
    b200.update({"comm": comm, "device_resident_data": resident,
                 "wave_batched": os.environ.get("FLUTE_WAVE", "1") != "0"})
    if sync_ckpt:
        b200["async_checkpoint"] = False
    if task == "cv_resnet_fedcifar100":
        raw["model_config"]["group_norm"] = 2 if norm == "gn" else 0
    if compute_dtype or spec.get("dtype"):
        raw["model_config"]["compute_dtype"] = compute_dtype or spec["dtype"]
    for section, upd in (spec.get("overrides") or {}).items():
        tgt = raw
        keys = section.split(".")
        for k in keys[:-1]:
            tgt = tgt.setdefault(k, {})
        if isinstance(upd, dict) and isinstance(tgt.get(keys[-1]), dict):
            tgt[keys[-1]].update(upd)
        else:
            tgt[keys[-1]] = upd
    return FLUTEConfig.from_dict(raw)


def build_job(task="cv_resnet_fedcifar100", n_clients_per_round=None, users=None, norm="gn", comm="auto", out_dir=None,
              resident=True, compute_dtype=None, sync_ckpt=False):
    import tempfile
    from msrflute_b200 import cli
    config = make_config(task, n_clients_per_round, norm=norm, comm=comm, resident=resident,
                         compute_dtype=compute_dtype, sync_ckpt=sync_ckpt)
    out_dir = out_dir or tempfile.mkdtemp(prefix="flute_bench_")
    model_path = os.path.join(out_dir, "models")
    os.makedirs(model_path, exist_ok=True)
    config["data_path"], config["output_path"], config["model_path"] = out_dir, out_dir, model_path
    config["experiment_name"] = "bench"
    config["client_config"]["task"] = task
    config["server_config"]["task"] = task
    config.validate()
    if users is not None and task == "cv_resnet_fedcifar100":          # smaller synthetic population (smoke tests)
        from msrflute_b200.utils.dataloaders_utils import get_exp_dataset
        from msrflute_b200.data import synthetic
        ds_cls = get_exp_dataset(task)
        ds_cls.synthetic_train = staticmethod(lambda: synthetic.make_image_classification(users, 100, (32, 32, 3), 100, seed=5))
        ds_cls.synthetic_test = staticmethod(lambda: synthetic.make_image_classification(max(users // 5, 2), 100, (32, 32, 3), 100, seed=6))
    server, worker, comm_obj = cli.build_job(config, task, out_dir, model_path)
    return BenchJob(server, worker, comm_obj, config)


def build_flagship(n_clients_per_round=10, users=None, norm="gn", comm="auto", out_dir=None, resident=True,
                   compute_dtype="fp32"):
    return build_job("cv_resnet_fedcifar100", n_clients_per_round, users=users, norm=norm, comm=comm, out_dir=out_dir,
                     resident=resident, compute_dtype=compute_dtype)


def _settle(server, cuda, torch, max_rounds=40, tol=0.05, fixed=None):
    """Set-up rounds (not warm-up): run until two consecutive rounds agree within ``tol`` — CUDA-graph capture on every
    rank, symmetric-memory peer mappings and signal pads, NCCL channel set-up and allocator growth happen here.
    ``fixed`` runs exactly that many rounds instead, so the model the later rounds start from does not depend on timing."""
    import time
    if fixed is not None:
        server.run_rounds(fixed)
        return fixed
    prev, n = None, 0
    while n < max_rounds:
        if cuda:
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        server.run_rounds(1)
        if cuda:
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        n += 1
        if prev is not None and n >= 4 and abs(dt - prev) <= tol * max(dt, prev):
            break
        prev = dt
    return n


def _restore_global_model(server, snapshot):
    """Copies ``snapshot`` back into the global model in place (its tensors are views of the weight arena that the
    captured CUDA graphs read) and makes the next round resend the weights to the workers."""
    import torch
    with torch.no_grad():
        for k, v in server.worker_trainer.model.state_dict().items():
            v.copy_(snapshot[k])
    server._weights_in_sync = False


def _dump_outputs(out_dir, server, loss):
    """``--dump-outputs``: the last round's train loss and the global model it left behind, as ``out_dir/<name>.npy``."""
    import numpy as np
    import torch
    sd = server.worker_trainer.model.state_dict()
    flat = torch.cat([t.detach().reshape(-1).float() for t in sd.values() if t.is_floating_point()])
    if flat.numel() > DUMP_MAX_VALUES:
        idx = np.unique(np.random.default_rng(0).integers(0, flat.numel(), DUMP_MAX_VALUES))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "global_model.npy"), flat.cpu().numpy())
    np.save(os.path.join(out_dir, "train_loss.npy"), np.asarray([float("nan") if loss is None else float(loss)], np.float64))


def main():
    args = parse_args()
    if args.impl == "reference":
        _reference(args)
        return
    import logging
    import statistics
    import time
    import torch
    if args.dump_outputs:
        args.dump_outputs = os.path.abspath(args.dump_outputs)
    os.chdir(ROOT)
    logging.getLogger().setLevel(logging.WARNING)
    spec = TASKS[args.task]
    cpu_dry_run = os.environ.get("FLUTE_BENCH_CPU") == "1"       # control-flow test of the multi-rank protocol (gloo)
    if not torch.cuda.is_available() and not cpu_dry_run:
        emit({"metric": spec["metric"], "value": None, "unavailable": "no CUDA device"})
        return
    cuda = torch.cuda.is_available()
    from msrflute_b200.ops import _ext
    from msrflute_b200.utils.timing import PHASES
    if cuda:
        _ext.load(required=True)
    from msrflute_b200.core.federated import Server
    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    cpr = args.clients_per_round or spec["clients_per_round"]
    job = build_job(args.task, cpr, users=(20 if cpu_dry_run else None), norm=args.norm, comm=args.comm,
                    compute_dtype=os.environ.get("FLUTE_BENCH_DTYPE") or None, sync_ckpt=args.sync_ckpt)
    comm = job.comm
    eng = getattr(job.worker, "engine", None)
    do_e2e = not args.no_e2e and (eng is not None or cpu_dry_run)

    if rank != 0:
        # Workers live in the command loop; the server brackets the timed regions with sync_nodes() (every rank
        # drains its GPU, records a CUDA event, then barriers), so each rank knows its own device time per region.
        job.worker.run()
        w = job.worker
        ms = w.sync_region_ms(0, 1) if cuda else 0.0
        phases = PHASES.totals() if cuda else {}
        comm.gather_objects({"ms": ms, "phases": phases,
                             "h2d": int(getattr(w.engine, "h2d_bytes_last_round", 0) or 0)})
        comm.close()
        return

    server = job.server
    server.begin_training()
    initial_model = None
    if args.dump_outputs:
        initial_model = {k: v.detach().clone() for k, v in server.worker_trainer.model.state_dict().items()}
    setup_rounds = _settle(server, cuda, torch, fixed=SETUP_ROUNDS_FIXED if args.dump_outputs else None)
    server.run_rounds(args.warmup)
    Server.sync_nodes({"phases": True})                          # barrier + device synchronize on every rank
    PHASES.enable(True)
    sampler = ClockSampler(torch.cuda.current_device() if cuda else 0).start()
    n0 = _ext.LAUNCH_COUNTER["n"]
    marks = []
    if cuda:
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
        marks.append(e0)
    t0 = time.perf_counter()
    loss = None
    host_marks = [t0]
    for step in range(args.steps):
        if initial_model is not None and step == args.steps - 1:
            _restore_global_model(server, initial_model)
        loss = server.run_rounds(1)
        host_marks.append(time.perf_counter())
        if cuda:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append(ev)
    if os.environ.get("FLUTE_CKPT_TRACE") == "1":
        slow = sorted(range(args.steps), key=lambda i: -(host_marks[i + 1] - host_marks[i]))[:4]
        print("[bench] slowest host rounds: " + ", ".join("#{} {:.1f} ms ending t={:.3f}".format(
            i, (host_marks[i + 1] - host_marks[i]) * 1e3, host_marks[i + 1]) for i in slow), flush=True)
    Server.sync_nodes({"phases": False})
    t1 = time.perf_counter()
    clocks = sampler.stop()
    launches = _ext.LAUNCH_COUNTER["n"] - n0
    wall_ms = (t1 - t0) * 1e3
    dev_ms = marks[0].elapsed_time(marks[-1]) if cuda else wall_ms
    per_round = [marks[i].elapsed_time(marks[i + 1]) for i in range(len(marks) - 1)] if cuda else []
    my_phases = PHASES.totals() if cuda else {}
    PHASES.enable(False)
    if args.dump_outputs:
        _dump_outputs(args.dump_outputs, server, loss)

    # End-to-end variant: every engine streams its clients' shards host(pinned)->device inside the timed region and the
    # per-round record table is read back (it always is); timed by wall clock around the public run_rounds() call.
    e2e = None
    if do_e2e:
        Server.sync_nodes({"resident": False})                  # engines keep the pack in pinned host memory
        server.run_rounds(3)                                    # settle
        Server.sync_nodes()
        t2 = time.perf_counter()
        server.run_rounds(args.steps)
        Server.sync_nodes()
        e2e_s = time.perf_counter() - t2
        e2e = {"value": args.steps / e2e_s, "unit": "rounds/s",
               "h2d_bytes_per_step": int(getattr(eng, "h2d_bytes_last_round", 0) or 0),
               "d2h_bytes_per_step": int(getattr(eng, "d2h_bytes_last_round", 0) or 0),
               "note": "wall clock incl. host orchestration, checkpoint snapshots, H2D of the sampled clients' "
                       "shards from pinned memory and D2H of the per-round loss/statistics table (rank 0's bytes; "
                       "all ranks stream their own shards)"}
    server.end_training()
    ms = max(dev_ms, 0.0)
    rank_ms = None
    phase_sets = [my_phases]
    if comm.size > 1:
        others = [o for o in comm.gather_objects({"ms": ms}) if isinstance(o, dict)]
        rank_ms = [round(float(o.get("ms", 0.0)), 3) for o in others]
        ms = max([ms] + [o.get("ms", 0.0) for o in others])
        phase_sets += [o.get("phases") or {} for o in others if "phases" in o]
        if e2e is not None:
            e2e["h2d_bytes_per_step"] += sum(int(o.get("h2d", 0)) for o in others)
    value = args.steps / (ms / 1e3)

    # exposed model-distribution + gather time per round: per phase the max over ranks, then summed
    names = sorted({k for ps in phase_sets for k in ps})
    per_phase = {k: max(ps.get(k, 0.0) for ps in phase_sets) / args.steps for k in names}
    exposed = sum(per_phase.values())
    arena_bytes = 0
    try:
        from msrflute_b200.parallel.arena import module_arena
        arena_bytes = int(module_arena(server.worker_trainer.model)[0].flat.numel()) * 4
    except Exception:
        pass
    comm_info = {"ms_per_round": round(exposed, 4), "phases_ms_per_round": {k: round(v, 4) for k, v in per_phase.items()},
                 "note": "device time of slot scatter-in (bcast_local), fused pseudo-gradient accumulation (gather_local), "
                         "cross-GPU reduce (gather_xgpu) and fused reduce+update+broadcast kernel with its barriers "
                         "(update_bcast); one stream, so none of it overlaps client compute"}
    if world > 1 and arena_bytes:
        ideal_ms = (world - 1) * arena_bytes / 770e9 * 1e3       # in and out of the server GPU concurrently
        xg = per_phase.get("gather_xgpu", 0.0) + per_phase.get("update_bcast", 0.0) + per_phase.get("bcast_xgpu", 0.0)
        comm_info.update({"xgpu_ms_per_round": round(xg, 4), "nvlink_roofline_ms": round(ideal_ms, 4),
                          "fraction_of_nvlink_roofline": round(ideal_ms / xg, 3) if xg > 0 else None,
                          "roofline": "(N-1) x {} B arena each way through rank 0's links at the measured 770 GB/s per "
                                      "direction".format(arena_bytes)})
    med = statistics.median(per_round) if per_round else None
    emit({
        "metric": spec["metric"], "value": value, "unit": "rounds/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "wall_ms_per_step": wall_ms / args.steps,
        "median_ms_per_round": med, "rounds_per_s_at_median": (1e3 / med) if med else None,
        "round_ms_min_max": [round(min(per_round), 3), round(max(per_round), 3)] if per_round else None,
        "slowest_rounds": sorted(([i, round(v, 2)] for i, v in enumerate(per_round)), key=lambda t: -t[1])[:5],
        "setup_rounds": setup_rounds,
        "higher_is_better": True, "scaling": "strong",
        "vs_baseline": (value / BASELINE_PUBLISHED[args.task]) if BASELINE_PUBLISHED.get(args.task) else None,
        "dtype": spec.get("dtype_label", "fp32 storage, tf32 tensor-core math (tcgen05 kind::tf32)"),
        "data": spec["data"], "clocks": clocks, "e2e": e2e, "exposed_comm": comm_info,
        "gpu_launches": int(launches), "impl": "ours", "last_train_loss": loss,
        "rank_ms": rank_ms if comm.size > 1 else None,
        "config": dict(spec["config"], clients_per_round=cpr,
                       norm=(args.norm if args.task == "cv_resnet_fedcifar100" else None),
                       parallelism="fl-clients-over-{}gpu(s), {} transport".format(world, comm.kind),
                       l2="no explicit flush: every round streams the per-client weight / gradient arenas (> 126 MB L2 "
                          "for the flagship) and re-samples clients",
                       checkpoint=("latest_model.tar written synchronously every round (reference behaviour)"
                                   if args.sync_ckpt else
                                   "latest_model.tar snapshot every round (async writer, latest-wins, <=0.25 s stale)")),
    })
    comm.close()


if __name__ == "__main__":
    main()
