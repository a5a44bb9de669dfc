"""Helpers shared by both benchmark arms (self-contained: imports nothing from msrflute_b200)."""
import argparse
import json
import os
import statistics
import subprocess
import threading
import time

HEADLINE_METRIC = "fl_rounds_per_sec_resnet18_fedcifar100"
BASELINE_PUBLISHED_ROUNDS_PER_SEC = 4000.0 / 6121.0     # BASELINE.md: RESNET_FEDCIFAR100, 4000 rounds in 01:42:01

#: rounds/s derived from the reference's published time-to-finish tables (BASELINE.md); None = nothing published
BASELINE_PUBLISHED = {
    "cv_resnet_fedcifar100": 4000.0 / 6121.0,
    "cv_cnn_femnist": 1500.0 / 502.0,
    "nlp_rnn_fedshakespeare": 1200.0 / 1310.0,
    "cv_lr_mnist": 100.0 / 95.0,
    "mlm_bert": None,
}

#: the BASELINE.json configs: metric name, clients per round, data description, config block of the JSON line and
#: config overrides applied on top of experiments/<task>/config.yaml
TASKS = {
    "cv_resnet_fedcifar100": {
        "metric": HEADLINE_METRIC, "clients_per_round": 10, "dtype": "fp32",
        "dtype_label": "fp32 storage, tf32 tensor-core math (tcgen05 kind::tf32)",
        "data": "synthetic Fed-CIFAR-100 shape (500 users x 100 x 32x32x3 uint8), random-init weights",
        "config": {"model": "ResNet-18 (GroupNorm 2 ch/group, per-group affine; 1000-way FC like the reference's RESNET), "
                            "11.7M params", "client_batch": 20, "local_steps_per_client": 5, "global_batch": 1000,
                   "seq_len": None},
    },
    "cv_cnn_femnist": {
        "metric": "fl_rounds_per_sec_cnn_femnist", "clients_per_round": 10,
        "dtype_label": "bf16 autocast (compute_dtype: bf16 of the task config), fp32 master weights / optimizer",
        "data": "synthetic FedEMNIST shape (3400 users x ~100 x 28x28 uint8, 62 classes), random-init weights",
        "config": {"model": "CNN_DropOut (2 conv + 2 FC, 1.2M params)", "client_batch": 20, "global_batch": None,
                   "seq_len": None},
    },
    "nlp_rnn_fedshakespeare": {
        "metric": "fl_rounds_per_sec_rnn_fedshakespeare_quantized_gather", "clients_per_round": 10,
        "dtype_label": "fp32 (persistent LSTM kernels, fp32 FMA); 8-bit quantised pseudo-gradients on the gather path",
        "data": "synthetic Shakespeare shape (715 users x sequences of 80 tokens, vocab 90), random-init weights",
        "config": {"model": "Embedding(90,8) + 2xLSTM(256) + FC(90), 0.82M params; DGA with 8-bit gradient "
                            "quantization on the gather path", "client_batch": 4, "global_batch": None, "seq_len": 80},
        "overrides": {"strategy": "DGA", "server_config.aggregate_median": "mean",
                      "client_config.quant_thresh": 0.5, "client_config.quant_bits": 8, "client_config.quant_anneal": 1.0},
    },
    "mlm_bert": {
        "metric": "fl_rounds_per_sec_bert_base_mlm_global_dp", "clients_per_round": 32,
        "dtype_label": "fp32 master weights; bf16 tensor-core GEMMs and attention (tcgen05 kind::f16), fp32 accumulate",
        "data": "synthetic token blobs (1000 users, max_seq_length 128, vocab 30522), random-init BERT-base",
        "config": {"model": "BERT-base MLM (HF config, 110M params), DGA + global DP", "client_batch": 8,
                   "global_batch": None, "seq_len": 128},
    },
    "cv_lr_mnist": {
        "metric": "fl_rounds_per_sec_lr_mnist", "clients_per_round": 10,
        "data": "synthetic MNIST shape (1000 users x 784), random-init weights",
        "config": {"model": "logistic regression 784x10", "client_batch": 10, "global_batch": None, "seq_len": None},
    },
}


def parse_args(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=None, help="timed rounds (default: 200 for this repo's flagship — a "
                   "1.3 s timed region —, 40 for the other tasks, 20 for the reference arm, whose rounds take seconds)")
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--task", default="cv_resnet_fedcifar100", choices=sorted(TASKS))
    p.add_argument("--norm", default="gn", choices=["gn", "bn"], help="ours only: GroupNorm (BASELINE.json) or "
                   "BatchNorm (what the reference actually instantiates)")
    p.add_argument("--comm", default="auto")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--clients-per-round", type=int, default=None, help="default: the BASELINE config's value")
    p.add_argument("--sync-ckpt", action="store_true", help="ours only: write latest_model.tar synchronously every "
                   "round like the reference (default: async latest-wins writer)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None, help="ours only: after the timed rounds write the "
                   "last one's results (train loss, global model) to DIR/<name>.npy; set-up then runs a fixed number "
                   "of rounds so the inputs of every round are the same on every run")
    args = p.parse_args(argv)
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else (200 if args.task in ("cv_resnet_fedcifar100", "cv_lr_mnist") else 40)
    return args


class ClockSampler:
    """Samples ``nvidia-smi`` SM clocks + throttle reasons while the timed region runs (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0, period_ms=100):
        self.gpu, self.period = gpu_index, period_ms
        self.proc, self.lines = None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", str(self.period)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._read, daemon=True)
            self._t.start()
        except (OSError, FileNotFoundError):
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def emit(d):
    print(json.dumps(d), flush=True)
