#!/usr/bin/env python
"""bench.py -- the benchmark of carla_ppo_b200.

    python bench.py --gpus N --steps K --warmup W            (this build: sm_100a CUDA behind the C ABI)
    python bench.py --steps K --warmup W --dump-outputs DIR  (also write what the last timed step computed, see below)
    python bench.py --impl reference --steps K --warmup W    (the reference's CPU path on the host cores)
    python bench.py --config 5 [--gpus N]                    (BASELINE configs[4]: 100 k frames -> encode -> PPO loop)

Metric (BASELINE.json): VAE frames/sec @ batch 4096 -- one "step" is one ConvVAE train step (forward +
MSE/KL loss + backward + TF-Adam, parameters updated in place) on synthetic 160x80x3 frames, z_dim 64
(BASELINE configs[1]); N>1 shards the SAME global batch of 4096 frames over N ranks (configs[3], strong
scaling) with one NCCL all-reduce of the flat gradient per step.  Secondary object "ppo": the PPO update
of configs[2] (T=2048 rollout, 4 epochs x 256 minibatch, shipped agent checkpoint-705) in latent-updates/sec.

One JSON line on stdout (rank 0).  Keys follow the contract:
  value        whole-job frames/s with inputs resident in HBM (CUDA events, max over ranks);
  e2e          the same step fed from pinned HOST buffers through the public host-fed API, H2D of the frames and D2H of
               the losses inside the timed region: `e2e.value` is ConvVAE.train_step_async (input prefetch on a copy
               stream, torch copies + cpb_vae_loss_grad + cpb_adam_apply_guarded), `e2e.sync_host` is the plain C entry
               cpb_vae_train_step_host (blocking copy -> step -> read-back, what the reference's feed_dict does);
  roofline     dominant kernel group vs MEASURED peaks (MEASURED_PEAKS.json for HBM / bf16; the TF32 tensor and fp32 FMA
               peaks are measured here, BASELINE.md section 3) + per-group device times on rank 0 (also for N>1);
  dp_check     (N>1) replicas bit-identical after the timed steps, N-rank loss / gradient vs a 1-rank recompute;
  cpu_baseline torch-CPU fp32 restatement of the reference graph ("port": TensorFlow 1.13 cannot be installed).

--steps K is the number of steps of every timed loop (device-resident, host-fed, blocking host entry, PPO learn()).
--dump-outputs DIR (rank 0) writes, as DIR/<name>.npy in float32, what a caller of each timed path holds after its last
timed call: vae_losses ([recon, kl] the step returns), vae_params.<tensor> (the parameters it updated in place) and
vae_grads.<tensor> (the gradient that update used); ppo_metrics (the per-minibatch losses of the last learn()) and
ppo_params.<tensor> (N=1 only).  Tensor names are the reference's variable names with '/' -> '.'.  The inputs and
weights are seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

GLOBAL_BATCH = 4096
Z_DIM = 64
FLOP_PER_FRAME_TRAIN = 776_494_080          # SURVEY.md section 8(d)
BYTES_PER_FRAME_TRAIN = 10_164_000           # layer-materialised fp32 model, SURVEY.md section 8(d)

# algorithmic MACs per frame of each labelled kernel group (SURVEY appendix A.1; x2 for FLOPs)
MAC = {"conv1": 4_732_416, "conv2": 22_413_312, "conv3": 18_874_368, "conv4": 12_582_912,
       "heads": 786_432, "dense1": 393_216, "deconv1": 12_582_912, "deconv2": 18_874_368,
       "deconv3": 35_020_800, "deconv4": 4_732_416}

DUMP_LIMIT_BYTES = 64 << 20


def tensor_dumps(prefix, tensors):
    """{'<prefix>.<name with / -> .>': float32 array} of a name -> array dict (get_weights() / get_grads())."""
    return {"%s.%s" % (prefix, k.replace("/", ".")): np.asarray(v, np.float32) for k, v in tensors.items()}


def write_dumps(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy, refusing a set larger than DUMP_LIMIT_BYTES."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def kernel_source_hash():
    """sha256 over the CUDA sources: the committed ncu traffic table is only valid for the sources it was captured from."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "carla_ppo_b200", "csrc")
    for fn in sorted(os.listdir(d)):
        if fn.endswith((".cu", ".cuh")):
            with open(os.path.join(d, fn), "rb") as f:
                h.update(fn.encode()); h.update(f.read())
    return h.hexdigest()[:16]


def load_ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of each labelled kernel group, extracted from the committed
    `ncu --set full` capture by scripts/ncu_traffic.py into profiles/r2_ncu_traffic.json together with the hash of the
    sources it was captured from -- so a kernel change that is not re-profiled shows up as `traffic_stale`."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if not os.path.isfile(path):
        return {}, None
    with open(path) as f:
        t = json.load(f)
    return t.get("bytes_per_launch", {}), t.get("source_hash")


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_burst=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def measure_fp32_peaks(seconds=0.6):
    """BASELINE.md section 3: the fp32-FMA and TF32 tensor peaks are measured in the harness (MEASURED_PEAKS.json has only
    HBM and bf16).  cuBLAS GEMMs 8192^3, best of the repetitions that fit `seconds`; measurement only, not the product path."""
    import torch
    n = 8192
    a = torch.randn(n, n, device="cuda"); b = torch.randn(n, n, device="cuda")
    out = {}
    old = torch.backends.cuda.matmul.allow_tf32
    try:
        for key, tf32 in (("fp32_fma_tflops", False), ("tf32_tflops", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.matmul(a, b); torch.cuda.synchronize()
            best, t_end = 0.0, time.perf_counter() + seconds
            while time.perf_counter() < t_end:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
                best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
            out[key] = best
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    out["how"] = "torch.matmul fp32 8192^3, allow_tf32 off / on, best CUDA-event time"
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ================================================================================================== ours
def make_vae(model_dir, data_parallel):
    from carla_ppo_b200.vae.models import ConvVAE
    vae = ConvVAE((80, 160, 3), z_dim=Z_DIM, beta=1.0, learning_rate=1e-4, loss_fn="mse", model_dir=model_dir,
                  seed=0, data_parallel=data_parallel)
    vae.init_session(init_logging=False)          # glorot-uniform random init of the reference architecture (seed 0)
    return vae


def profile_groups(lib, vae, x, eps, steps, enabled=True):
    """Per-call-site device time (CUDA events on the launching stream) over `steps` extra steps.  Under N>1 every rank
    runs the steps (they contain the all-reduce); only rank 0 (`enabled`) records."""
    import torch
    if enabled:
        lib.cpb_profile_reset(); lib.cpb_profile_enable(1)
    for _ in range(steps):
        vae.train_step_device(x, x, eps)
    torch.cuda.synchronize()
    if not enabled:
        return {}
    lib.cpb_profile_enable(0)
    buf = C.create_string_buffer(1 << 16)
    n = lib.cpb_profile_report(buf, len(buf))
    lib.cpb_profile_reset()
    groups = {}
    for line in buf.raw[:n].decode().splitlines():
        label, count, ms = line.split()
        groups[label] = {"launch_groups": int(count) // 1, "ms_per_step": float(ms) / steps}
    return groups


PPO_FLOP_PER_LEARN = 20.0e9        # SURVEY section 8(d): 2.44 MFLOP per sample-step x 2048 x 4
PPO_BYTES_PER_LEARN = 0.35e9


def ppo_config3_inputs():
    """SURVEY section 8(d) config 3 (= tests/test_ppo_gpu.py::_baseline_config3)."""
    T, E = 2048, 4
    rs = np.random.RandomState(0)
    states = rs.randn(T, 67).astype(np.float32)
    actions = np.clip(rs.randn(T, 2), [-1.0, 0.0], [1.0, 1.0]).astype(np.float32)
    rewards = rs.rand(T); values = rs.randn(T).astype(np.float32)
    dones = np.zeros(T, bool); dones[-1] = True
    prs = np.random.RandomState(0)
    perms = np.stack([prs.permutation(T) for _ in range(E)])
    return states, actions, rewards, values, dones, perms


def shipped_agent():
    z = np.load(os.path.join(ROOT, "tests", "golden", "ppo_ckpt705.npz"))
    names = ["dense/kernel", "dense/bias", "dense_1/kernel", "dense_1/bias", "action_mean/kernel", "action_mean/bias", "action_logstd",
             "dense_2/kernel", "dense_2/bias", "dense_3/kernel", "dense_3/bias", "value/kernel", "value/bias"]
    return ({k: z["policy/" + k] for k in names}, {k: z["policy_old/" + k] for k in names}, {k: z["adam_m/" + k] for k in names},
            {k: z["adam_v/" + k] for k in names}, (float(z["beta1_power"]), float(z["beta2_power"])))


def bench_ppo(lib, steps=10, cpu=True, dumps=None):
    """BASELINE configs[2]: T=2048 rollout of 67-d states, 4 epochs x 8 minibatches of 256, weights = the reference's shipped
    agent checkpoint-705 (policy, policy_old, warm Adam slots); timed: GAE + normalisation + theta_old copy + 32 Adam steps.
    `dumps` (a dict) receives the metrics and parameters of the last timed learn()."""
    import torch
    from carla_ppo_b200.ppo import PPO

    class Box:
        low = np.array([-1.0, 0.0], np.float32); high = np.array([1.0, 1.0], np.float32); shape = (2,)
    pol, old, am, av, pw = shipped_agent()
    ppo = PPO((67,), Box(), learning_rate=1e-4, value_scale=1.0, entropy_scale=0.01, epsilon=0.2, model_dir=tempfile.mkdtemp(), seed=0)
    ppo.init_session(init_logging=False)
    ppo.set_weights(pol, old, am, av, pw)
    T, E, B = 2048, 4, 256
    s_, a_, r_, v_, d_, perms_ = ppo_config3_inputs()
    dev = ppo._device
    s = torch.from_numpy(s_).to(dev); a = torch.from_numpy(a_).to(dev)
    r = torch.from_numpy(r_).to(dev); v = torch.from_numpy(v_.astype(np.float64)).to(dev)
    d = torch.from_numpy(d_.astype(np.float64)).to(dev)
    perms = torch.from_numpy(perms_.astype(np.int32)).to(dev)
    for _ in range(3):
        ppo.learn(s, a, v, r, d, 0.3, num_epochs=E, batch_size=B, perms=perms)
    torch.cuda.synchronize()
    lib.cpb_reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ppo.learn(s, a, v, r, d, 0.3, num_epochs=E, batch_size=B, perms=perms)
    e1.record(); torch.cuda.synchronize()
    if dumps is not None:
        dumps["ppo_metrics"] = ppo._pending_metrics[-1].cpu().numpy()
        dumps.update(tensor_dumps("ppo_params", ppo.get_weights()))
    ms = e0.elapsed_time(e1) / steps
    launches = int(lib.cpb_launch_count()) // steps
    out = {"metric": "PPO latent-updates/sec", "value": T * E / ms * 1e3, "unit": "sample-updates/s", "ms_per_learn": ms,
           "learn_calls_per_s": 1e3 / ms, "gpu_launches_per_learn": launches,
           "config": {"workload": "T=2048 rollout x 67-d states, 4 epochs x 8 minibatches of 256, GAE+normalise+theta_old copy+32 Adam steps",
                      "weights": "reference agent checkpoint-705 (policy, policy_old, Adam m/v, beta powers) from tests/golden/ppo_ckpt705.npz"},
           "floor": {"note": "neither roofline binds (SURVEY 8d): 20 GFLOP and 0.35 GB per learn(); the floor is launch / dependency latency",
                     "fp32_fma_ms": None, "hbm_ms": PPO_BYTES_PER_LEARN / (load_peaks()["hbm_gbs"] * 1e9) * 1e3,
                     "launch_floor_ms": launches * 2.0e-3,
                     "launch_floor_note": "launches x ~2 us back-to-back launch latency of a dependent chain"}}
    if cpu:
        from oracle.torch_ref import TorchPPOLearner
        tl = TorchPPOLearner(pol, Box.low, Box.high, lr=1e-4, epsilon=0.2, value_scale=1.0, entropy_scale=0.01)
        best, best_t = None, float("inf")
        tried = {}
        for c in sorted({1, 4, 8, 16, min(32, os.cpu_count() or 1)}):
            torch.set_num_threads(c)
            tl.learn(s_, a_, v_, r_, d_, 0.3, 0.99, 0.95, 1, B, perms_)
            t0 = time.perf_counter(); tl.learn(s_, a_, v_, r_, d_, 0.3, 0.99, 0.95, 1, B, perms_); dt = time.perf_counter() - t0
            tried[str(c)] = round(dt * 1e3, 2)
            if dt < best_t:
                best, best_t = c, dt
        torch.set_num_threads(best)
        n, t0 = 0, time.perf_counter()
        while n < 3 or (time.perf_counter() - t0 < 3.0 and n < 20):
            tl.learn(s_, a_, v_, r_, d_, 0.3, 0.99, 0.95, E, B, perms_); n += 1
        cpu_ms = (time.perf_counter() - t0) / n * 1e3
        out["cpu_baseline"] = {"value": T * E / cpu_ms * 1e3, "unit": "sample-updates/s", "ms_per_learn": cpu_ms, "cores": best, "kind": "port",
                               "threads_tried_ms_per_epoch": tried,
                               "sample": "%d full learn() calls of the same rollout (torch-CPU fp32 restatement of train.py:171-207 + ppo.py)" % n}
    return out


def pick_cpu_threads(make_step, candidates=None):
    """The GPU boxes expose 128 logical CPUs shared with other tenants; oneDNN on all of them is often far slower
    than on a subset.  Time one step per candidate thread count and keep the fastest ("all the host threads it can
    use" = as many as actually help)."""
    import torch
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = candidates or sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], float("inf")
    tried = {}
    for c in cands:
        torch.set_num_threads(c)
        make_step()                      # warm-up at this thread count
        t0 = time.perf_counter(); make_step(); dt = time.perf_counter() - t0
        tried[str(c)] = round(dt * 1e3, 1)
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    pick_cpu_threads.last = {"logical_cpus": ncpu, "ms_per_64_frame_step_by_threads": tried, "chosen": best}
    return best


def cpu_baseline_vae(seconds=12.0, micro=256):
    """torch-CPU fp32 restatement of the reference train step on a bounded sample (micro-batches of 256)."""
    import torch
    from oracle.torch_ref import TorchVAETrainer
    from oracle.vae_oracle import glorot_init
    tr = TorchVAETrainer(glorot_init(0), lr=1e-4, loss_type="mse")
    g = torch.Generator(); g.manual_seed(0)
    x = torch.rand(micro, 80, 160, 3, generator=g); eps = torch.randn(micro, Z_DIM, generator=g)
    xs, es = x[:64], eps[:64]
    pick_cpu_threads(lambda: tr.step(xs, xs, es))
    tr.step(x, x, eps)                                   # warm-up
    n = 0
    t0 = time.perf_counter()
    while True:
        tr.step(x, x, eps); n += 1
        dt = time.perf_counter() - t0
        if dt >= seconds or n >= 64:
            break
    return {"value": n * micro / dt, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
            "thread_calibration": getattr(pick_cpu_threads, "last", None),
            "sample": "%d full train steps (fwd+loss+bwd+TF-Adam) on micro-batches of %d synthetic frames, torch-CPU fp32 "
                      "restatement of the TF-1.13 graph (TensorFlow itself is not installable here)" % (n, micro)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from carla_ppo_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    # the contract is ONE JSON line on stdout: anything native libraries print meanwhile (NCCL's version banner, with
    # NCCL_DEBUG=INFO its whole log) is sent to stderr by pointing fd 1 at fd 2 until the line is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    assert GLOBAL_BATCH % world == 0
    B = GLOBAL_BATCH // world
    tmp = tempfile.mkdtemp()
    vae = make_vae(tmp, data_parallel=world > 1)
    g = torch.Generator(device="cuda"); g.manual_seed(1234 + rank)
    x = torch.rand(B, 80, 160, 3, generator=g, device="cuda")            # 629 MB at B=4096: larger than the 126 MB L2
    eps = torch.randn(B, Z_DIM, generator=g, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        vae.train_step_device(x, x, eps)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.cpb_reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        vae.train_step_device(x, x, eps)
    e1.record()
    barrier()
    dumps = None
    if args.dump_outputs and rank == 0:
        # copied before anything else runs: the e2e and profiling steps below keep training the same model
        dumps = {"vae_losses": vae._losses.cpu().numpy()}
        dumps.update(tensor_dumps("vae_params", vae.get_weights()))
        dumps.update(tensor_dumps("vae_grads", vae.get_grads()))
    launches = int(lib.cpb_launch_count())
    elapsed = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(elapsed, op=dist.ReduceOp.MAX)
    ms_step = float(elapsed.item()) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    value = GLOBAL_BATCH / ms_step * 1e3

    # ---- e2e: the same step fed from pinned HOST memory through the public host-fed API
    xh = torch.empty(B, 80, 160, 3, dtype=torch.float32).pin_memory(); xh.copy_(x.cpu())
    eh = torch.empty(B, Z_DIM, dtype=torch.float32).pin_memory(); eh.copy_(eps.cpu())
    h2d = xh.numel() * 4 + eh.numel() * 4
    d2h = 12

    def e2e_run(nsteps):
        # input prefetch: H2D of step i+1 (copy stream) overlaps the compute of step i; every step's losses are read back
        # on the host (one step late)
        pending = None
        for _ in range(nsteps):
            h = vae.train_step_async(xh, None, eh)
            if pending is not None:
                pending.result()
            pending = h
        pending.result()
    e2e_steps = args.steps
    e2e_run(2); barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    barrier()
    e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = GLOBAL_BATCH / float(e2e_ms.item()) * 1e3

    # ---- e2e (N=1 only): the blocking C entry with HOST pointers, cpb_vae_train_step_host -- copy in, step, copy out,
    # stream synchronised inside the call, exactly how the reference's sess.run(feed_dict=...) behaves
    sync_host = None
    if world == 1:
        xn, en = xh.numpy(), eh.numpy()
        vae.train_step(xn, xn, en)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            vae.train_step(xn, xn, en)
        sh_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        sync_host = {"value": GLOBAL_BATCH / sh_ms * 1e3, "unit": "frames/s", "ms_per_step": sh_ms, "steps": e2e_steps,
                     "path": "ConvVAE.train_step(numpy) -> cpb_vae_train_step_host: cudaMemcpyAsync H2D (pinned source) -> train step -> "
                             "losses + verify_range flags D2H -> cudaStreamSynchronize, no overlap between steps"}

    # ---- N>1: data-parallel parity, visible to the driver (the 2-GPU pytest skips on a 1-GPU test box)
    dp_check = None
    if world > 1:
        ref = vae.params.clone(); dist.broadcast(ref, 0)
        same = torch.tensor([1 if torch.equal(ref, vae.params) else 0], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        # N-rank loss and gradient of the CURRENT parameters on the global batch ...
        vae.loss_grad_device(x, x, eps, 1.0 / world)
        dist.all_reduce(vae._gradbuf)
        dp_grad = vae.grads.clone(); dp_loss = vae._losses.clone()
        # ... against a 1-rank evaluation of the same global batch on rank 0 (every rank's shard is regenerated from its seed)
        if rank == 0:
            from carla_ppo_b200.vae.models import ConvVAE
            single = ConvVAE((80, 160, 3), z_dim=Z_DIM, beta=1.0, learning_rate=1e-4, loss_fn="mse", model_dir=tempfile.mkdtemp(), seed=0)
            single.init_session(init_logging=False)
            single.params.copy_(vae.params)
            xs, es = [], []
            for rk in range(world):
                gg = torch.Generator(device="cuda"); gg.manual_seed(1234 + rk)
                xs.append(torch.rand(B, 80, 160, 3, generator=gg, device="cuda")); es.append(torch.randn(B, Z_DIM, generator=gg, device="cuda"))
            xf, ef = torch.cat(xs), torch.cat(es)
            del xs, es
            single.loss_grad_device(xf, xf, ef)
            gerr = float((dp_grad.double() - single.grads.double()).norm() / single.grads.double().norm())
            lerr = float(((dp_loss.double() - single._losses.double()).abs() / single._losses.double().abs()).max())
            dp_check = {"replicas_bit_identical": bool(int(same.item())), "loss_rel_err_vs_1rank": lerr, "grad_rel_err_vs_1rank": gerr,
                        "ok": bool(int(same.item())) and lerr < 1e-5 and gerr < 1e-5,
                        "what": "after the timed steps: params of every rank == rank 0's (bitwise); [recon, kl] and the flat gradient of the "
                                "global batch from %d shards + all-reduce vs ONE cpb_vae_loss_grad over the 4096 frames on rank 0 "
                                "(norm-wise, bar 1e-5)" % world}
            del single, xf, ef
            torch.cuda.empty_cache()

    groups = profile_groups(lib, vae, x, eps, 3, enabled=(rank == 0))
    out = None
    if rank == 0:
        peaks = load_peaks()
        fp32_peaks = measure_fp32_peaks()
        traffic_tab, traffic_hash = load_ncu_traffic()
        roof = None
        if groups:
            # dominant = the labelled conv/deconv kernel group with the largest share of the step
            def flops(label):
                layer, kind = label.split(".")
                if layer not in MAC:
                    return 0.0
                return 2.0 * MAC[layer] * B
            conv_like = {k: v for k, v in groups.items() if "." in k and k.split(".")[0] in MAC}
            dom = max(conv_like, key=lambda k: conv_like[k]["ms_per_step"])
            ach = flops(dom) / (conv_like[dom]["ms_per_step"] * 1e-3) / 1e12
            total_ms = sum(v["ms_per_step"] for v in groups.values())
            mode = int(lib.cpb_get_math_mode())
            tc_ms = sum(v["ms_per_step"] for k, v in conv_like.items() if k.split(".")[0] not in ("conv1", "deconv4"))
            tc_flop = sum(flops(k) for k in conv_like if k.split(".")[0] not in ("conv1", "deconv4"))
            roof = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                    "frac": ach / peaks["bf16_sustained"],
                    "traffic": traffic_tab.get(dom) if world == 1 else None,
                    "traffic_source": "profiles/r2_ncu_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch at B=4096)",
                    "traffic_stale": (traffic_hash != kernel_source_hash()) if traffic_hash else None,
                    "share_of_step": conv_like[dom]["ms_per_step"] / total_ms,
                    "math_mode": "tcgen05 kind::tf32, 3xTF32 split (fp32-accurate)" if mode == 1 else "fp32 SIMT FMA",
                    "measured_peaks": {"tf32_tflops": fp32_peaks["tf32_tflops"], "fp32_fma_tflops": fp32_peaks["fp32_fma_tflops"], "how": fp32_peaks["how"],
                                       "bf16_tflops_sustained": peaks["bf16_sustained"], "hbm_gbs": peaks["hbm_gbs"], "source": peaks["source"]},
                    "frac_of_tf32_peak": ach / fp32_peaks["tf32_tflops"],
                    "frac_of_3xtf32_ceiling": ach / (fp32_peaks["tf32_tflops"] / 3.0),
                    "tensor_layers": {"ms_per_step": tc_ms, "achieved_tflops": tc_flop / (tc_ms * 1e-3) / 1e12,
                                      "frac_of_3xtf32_ceiling": tc_flop / (tc_ms * 1e-3) / 1e12 / (fp32_peaks["tf32_tflops"] / 3.0)},
                    "note": "achieved = algorithmic fp32-equivalent FLOPs of the layer / its CUDA-event time; peak = measured bf16 tensor figure "
                            "(contract); a 3xTF32 kernel issues 3 TF32 MMAs per algorithmic product, so its ceiling is the MEASURED TF32 peak / 3 "
                            "= %.0f TFLOP/s algorithmic" % (fp32_peaks["tf32_tflops"] / 3.0),
                    "step_hbm": {"bound": "hbm", "achieved": BYTES_PER_FRAME_TRAIN * GLOBAL_BATCH / (ms_step * 1e-3) / 1e9,
                                 "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": BYTES_PER_FRAME_TRAIN * GLOBAL_BATCH / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"]},
                    "groups_ms_per_step": {k: round(v["ms_per_step"], 4) for k, v in sorted(groups.items(), key=lambda kv: -kv[1]["ms_per_step"])}}
        cpu = cpu_baseline_vae() if (world == 1 and not args.no_cpu_baseline) else None
        ppo = bench_ppo(lib, steps=args.steps, cpu=not args.no_cpu_baseline, dumps=dumps) if world == 1 else None
        out = {"metric": "VAE frames/sec @ batch 4096", "value": value, "unit": "frames/s", "n_gpus": world,
               "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {"workload": "ConvVAE train step (fwd + MSE/KL + bwd + TF-Adam), global batch 4096 x 160x80x3 -> 64-d latent "
                                      "(BASELINE configs[1]%s)" % ("" if world == 1 else "; configs[3]: sharded %d/GPU, one NCCL all-reduce of the flat gradient" % B),
                          "global_batch": GLOBAL_BATCH, "per_gpu_batch": B, "z_dim": Z_DIM, "loss": "mse", "lr": 1e-4,
                          "weights": "glorot-uniform random init (reference architecture)",
                          "l2": "inputs (629 MB/step at N=1) and activations (GBs) exceed the 126 MB L2; no explicit flush"},
               "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                       "ms_per_step": float(e2e_ms.item()), "steps": e2e_steps,
                       "path": "ConvVAE.train_step_async(host frames): pinned fp32 frames H2D on a copy stream (2 staging slots, "
                               "prefetch depth 1) -> cpb_vae_loss_grad (+NCCL all-reduce when N>1) -> cpb_adam_apply_guarded -> losses D2H every step",
                       "sync_host": sync_host},
               "gpu_launches": launches, "clocks": clocks, "algorithmic_tflops": FLOP_PER_FRAME_TRAIN * GLOBAL_BATCH / (ms_step * 1e-3) / 1e12}
        if roof:
            out["roofline"] = roof
        if dp_check:
            out["dp_check"] = dp_check
        if cpu:
            out["cpu_baseline"] = cpu
        if ppo:
            out["ppo"] = ppo
        if dumps is not None:
            write_dumps(args.dump_outputs, dumps)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(out), flush=True)
        os.dup2(2, 1)


# ============================================================================================= reference arm
def run_reference(args):
    """The reference's own CPU implementation of the path: torch-CPU fp32 restatement of the TF-1.13 graph
    (oracle/torch_ref.py, kind "port") with all host threads, each step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle.torch_ref import TorchVAETrainer
    from oracle.vae_oracle import glorot_init
    sample, micro = 512, 256
    tr = TorchVAETrainer(glorot_init(0), lr=1e-4, loss_type="mse")
    g = torch.Generator(); g.manual_seed(0)
    x = torch.rand(sample, 80, 160, 3, generator=g); eps = torch.randn(sample, Z_DIM, generator=g)
    pick_cpu_threads(lambda: tr.step(x[:64], x[:64], eps[:64]))
    for _ in range(max(1, min(args.warmup, 2))):
        tr.step(x, x, eps, micro_batch=micro)
    steps = max(1, min(args.steps, 20))
    t0 = time.perf_counter()
    for _ in range(steps):
        tr.step(x, x, eps, micro_batch=micro)
    dt = time.perf_counter() - t0
    value = steps * sample / dt
    desc = ("each step = one optimiser step on a bounded sample of %d synthetic frames (2 gradient-accumulation micro-batches "
            "of %d) instead of 4096; torch-CPU fp32 restatement of the reference's TF-1.13 graph (TensorFlow not installable)" % (sample, micro))
    print(json.dumps({"impl": "reference", "metric": "VAE frames/sec @ batch 4096", "value": value, "unit": "frames/s",
                      "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": steps, "warmup": max(1, min(args.warmup, 2)),
                      "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                      "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "ConvVAE train step (fwd + MSE/KL + bwd + TF-Adam), 160x80x3 -> 64-d latent; " + desc,
                                 "global_batch": GLOBAL_BATCH, "z_dim": Z_DIM, "loss": "mse", "lr": 1e-4},
                      "cpu_baseline": {"value": value, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port", "sample": desc},
                      "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", type=int, default=2, choices=[2, 5],
                    help="2 (default): the BASELINE metric, ConvVAE train step at batch 4096; 5: BASELINE configs[4], the offline "
                         "100k-frame encode -> PPO update pipeline (scripts/config5.py; frames sharded over the ranks)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != 2 or args.impl != "ours"):
        ap.error("--dump-outputs applies to the default benchmark (--impl ours --config 2)")
    if args.config == 5:
        import runpy
        sys.argv = [os.path.join(ROOT, "scripts", "config5.py")]
        runpy.run_path(sys.argv[0], run_name="__main__")
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
