"""bench.py -- ZMW windows/sec of the DeepConsensus model path on B200 (BASELINE.json metric).

  python bench.py --gpus 1 --steps K --warmup W            # the dcb200 engine
  python bench.py --impl reference --gpus 1 --steps K ...   # reference algorithm on host cores

A "step" is one pass of the hot path over one batch of synthetic pileup windows
(BASELINE.json configs[1]: 20 subreads x 120 bp, d_model 280, 6 layers, batch 1024 per GPU).
Multi-GPU (torchrun, one rank per GPU): windows are independent units, every rank scores its
own shard -- no data-path collective; NCCL carries only the barrier and the max-over-ranks
time reduction ("scaling": "weak").

value  : whole-job windows/s with the input rows already resident in HBM.
e2e    : the same metric through the reference-facing call with HOST buffers -- pinned-host rows are copied H2D
         and the base / quality characters copied D2H inside the timed region, every step.  `value` uses the
         pipelined C-ABI pair dcb_submit / dcb_wait exactly as inference.run_model_on_examples does (the copy of
         batch i+1 overlaps the kernels of batch i); `blocking_value` is dcb_forward one batch at a time.
roofline: tensor-core roofline of the dominant kernel (stack_pair_kernel: the whole encoder stack), timed with CUDA
         events on the engine's stream over K steps of the same workload (a separate pass: the `value` trials run
         with the per-kernel events off).  `frac` is against the BURST cuBLAS bf16 figure of MEASURED_PEAKS.json (the
         K-step region is tens of milliseconds); `roofline.sustained` repeats the measurement over >= 2 s of
         back-to-back steps against the sustained figure, with the clocks seen during it.
trials  : the K-step region is timed TRIALS (5) times, each bracketed by barrier + synchronize and reduced with MAX over
         ranks; `value` / `e2e` are the MEDIAN trial (all trials are listed).
parity  : the default (bf16 tensor-core) path against the engine's strict-fp32 path on the whole batch, on the
         device -- bases identical %, QV exact %, max |dQ|, max logit error (BASELINE.md section 3.4).
cpu_baseline / --impl reference: the oracle (torch-CPU fp32 restatement of the reference
         model, oracle/model.py) on the box's host cores.  This is the only place bench.py
         executes oracle/ -- as the baseline being reported, never as the product.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from deepconsensus_b200 import calibration as calibration_lib  # noqa: E402
from deepconsensus_b200 import params as params_lib            # noqa: E402
from deepconsensus_b200 import synthetic                       # noqa: E402
from deepconsensus_b200 import weights as weights_lib          # noqa: E402

METRIC = "zmw_windows_per_sec"
UNIT = "windows/s"
WORKLOAD = dict(workload="synthetic pileup windows (BASELINE configs[1])", max_passes=20,
                window=120, d_model=280, layers=6, heads=2, filter_size=2048, attn_win_size=12,
                batch_per_gpu=1024)
CALIBRATION = "0,1.197654,-0.99781"   # the fixture params.json's dc_calibration


def config_dict(world: int, batch: int):
  """The `config` of the JSON line -- identical for the engine arm and the --impl reference arm."""
  return dict(WORKLOAD, batch_per_gpu=batch, global_batch=batch * world,
              parallelism="dp%d (independent shards)" % world,
              l2="inputs larger than L2: the timed steps rotate over resident packed batches spanning > 126 MB of addresses, and "
                 "every step streams the 151 MB fp32 residual image through L2 (details under `timing`)")


def cpu_threads() -> int:
  """Threads of the CPU arm: the best count of a committed sweep on this pool's host (profiles/r02_cpu_sweep.json,
  scripts/cpu_sweep.py) when present, else every core the process may use."""
  avail = len(os.sched_getaffinity(0))
  path = os.path.join(ROOT, "profiles", "r02_cpu_sweep.json")
  if os.path.exists(path):
    try:
      with open(path) as f:
        best = int(json.load(f)["best_threads"])
      return max(1, min(best, avail))
    except Exception:
      pass
  return avail


def model_params():
  return params_lib.synthetic_params(max_passes=WORKLOAD["max_passes"], max_length=WORKLOAD["window"],
                                     num_hidden_layers=WORKLOAD["layers"])


def flops_per_window(p) -> float:
  """Algorithmic (un-padded, banded) FLOPs per window -- SURVEY.md section 8(d)."""
  L, d, ff, w = p.max_length, p.hidden_size, p.filter_size, p.attn_win_size
  E = params_lib.embedded_width(p)
  pairs = L * (2 * w + 1) - w * (w + 1)
  return 2 * L * E * d + p.num_hidden_layers * (8 * L * d * d + 4 * pairs * d + 4 * L * d * ff) + 2 * L * d * 5


def measured_peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    with open(path) as f:
      pk = json.load(f)
    return dict(bf16_tflops=pk["bf16_tflops"], bf16_tflops_sustained=pk.get("bf16_tflops_sustained"),
                hbm_gbs=pk["hbm_gbs"], source="MEASURED_PEAKS.json")
  return dict(bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, hbm_gbs=6650.0,
              source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
  """Samples nvidia-smi SM clock + throttle reasons for one GPU during the timed region."""

  def __init__(self, index: int):
    super().__init__(daemon=True)
    self.index, self.samples, self.stop_flag = index, [], threading.Event()
    self.max_mhz = None

  def run(self):
    q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    while not self.stop_flag.is_set():
      try:
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True,
                             timeout=5).stdout.strip().split(",")
        self.samples.append((float(out[0]), [o.strip() for o in out[2:]]))
        self.max_mhz = float(out[1])
      except Exception:
        pass
      self.stop_flag.wait(0.05)

  def summary(self):
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    if not self.samples:
      return dict(sm_mhz=None, sm_max_mhz=self.max_mhz, reasons=[], samples=0)
    reasons = sorted({names[i] for _, fl in self.samples for i, v in enumerate(fl) if v.lower().startswith("active")})
    return dict(sm_mhz=float(np.median([s[0] for s in self.samples])), sm_max_mhz=self.max_mhz,
                reasons=reasons, samples=len(self.samples))


def cpu_reference_windows_per_sec(p, w, sample_windows: int, reps: int, threads: int):
  """Times the oracle (reference algorithm restated on torch-CPU fp32) incl. argmax/QV."""
  import torch
  from oracle import model as omodel, postprocess as opost
  torch.set_num_threads(threads)
  rows = synthetic.make_rows(p, sample_windows, seed=99)
  cal = calibration_lib.parse_calibration_string(CALIBRATION)
  ts = []
  for _ in range(reps + 1):
    t = time.perf_counter()
    out = omodel.forward(rows, p, w)
    opost.quality_from_probs(out["probs"], 93, (cal.threshold, cal.w, cal.b))
    ts.append(time.perf_counter() - t)
  best = float(np.median(ts[1:])) if reps > 1 else ts[-1]
  return sample_windows / best, best


DUMP_LIMIT = 64 << 20   # bytes of all --dump-outputs files together


def dump_outputs(directory: str, **arrays):
  """--dump-outputs: each array (one row per window) as directory/<name>.npy in float32, so that two builds run with the
  same arguments can be compared output for output.  When the windows would exceed DUMP_LIMIT, the same fixed, seeded
  sample of windows is kept in every array and its indices are written as windows.npy (float64)."""
  arrays = {k: np.asarray(a, np.float32) for k, a in arrays.items()}
  n = len(next(iter(arrays.values())))
  per_window = sum(a.nbytes for a in arrays.values()) // max(n, 1) + 8
  keep = (DUMP_LIMIT - 4096) // per_window                      # 4 KB for the .npy headers
  if n > keep:
    idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    arrays = {k: a[idx] for k, a in arrays.items()}
    arrays["windows"] = idx.astype(np.float64)
  os.makedirs(directory, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(directory, name + ".npy"), a)


def run_reference(args, rank, world):
  """--impl reference: the reference's CPU path (oracle port) of the same workload on the host cores (rank 0 only).
  A step is the whole 1024-window batch, exactly as in the engine arm."""
  if rank != 0:
    return
  p = model_params()
  w = weights_lib.init_weights(p, seed=1)
  cores = cpu_threads()
  sample = args.batch
  import torch
  from oracle import model as omodel, postprocess as opost
  torch.set_num_threads(cores)
  rows = synthetic.make_rows(p, sample, seed=20240921 + 1)
  cal = calibration_lib.parse_calibration_string(CALIBRATION)

  def step():
    out = omodel.forward(rows, p, w)
    return opost.quality_from_probs(out["probs"], 93, (cal.threshold, cal.w, cal.b))
  for _ in range(args.warmup):
    step()
  t0 = time.perf_counter()
  for _ in range(args.steps):
    y, q = step()
  dt = time.perf_counter() - t0
  if args.dump_outputs:
    bases, quals = opost.to_ascii(y, q)
    dump_outputs(args.dump_outputs, bases=bases, quals=quals)
  value = sample * args.steps / dt
  desc = dict(value=value, unit=UNIT, cores=cores, kind="port",
              sample="%d synthetic windows per step (the full batch), torch-CPU fp32 oracle incl. argmax / QV" % sample)
  print(json.dumps(dict(metric=METRIC, value=value, unit=UNIT, impl="reference", n_gpus=args.gpus,
                        steps=args.steps, warmup=args.warmup, ms_per_step=dt / args.steps * 1e3,
                        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                        data="synthetic", config=config_dict(world, args.batch), cpu_baseline=desc,
                        e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))))


def bind_to_gpu_numa_node(index: int):
  """Best effort: run this rank (and therefore allocate its page-locked staging buffers) on the CPUs of the NUMA node
  the GPU hangs off, so the per-step host->device copies of 8 ranks do not cross the socket interconnect."""
  try:
    out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                         capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0].strip().lower()
    if out.startswith("00000000:"):
      out = out[4:]                      # sysfs uses a 4-digit PCI domain
    with open("/sys/bus/pci/devices/%s/numa_node" % out) as f:
      node = int(f.read().strip())
    if node < 0:
      return None
    with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
      cpus = set()
      for part in f.read().strip().split(","):
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    allowed = os.sched_getaffinity(0) & cpus
    if allowed:
      os.sched_setaffinity(0, allowed)
      return node
  except Exception:
    pass
  return None


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=200)
  ap.add_argument("--warmup", type=int, default=10)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--batch", type=int, default=WORKLOAD["batch_per_gpu"])
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--nccl-scatter", action="store_true",
                  help="N > 1: also time the step fed by ONE reader rank over NCCL (BASELINE configs[3]; secondary record, "
                       "profiles/r02_bench_{2,4,8}gpu.json were produced with it)")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="write the base and quality characters of the last timed step as DIR/bases.npy and DIR/quals.npy "
                       "(float32 [batch, window]; rank 0's shard when N > 1; a fixed sample of windows above 64 MB)")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  args.warmup = max(args.warmup, 3)

  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if args.impl == "reference":
    run_reference(args, rank, world)
    return

  import torch
  import torch.distributed as dist
  from deepconsensus_b200 import engine as engine_lib
  if not torch.cuda.is_available():
    raise SystemExit("bench.py: no CUDA device (the dcb200 engine has no CPU fallback)")
  torch.cuda.set_device(local)
  full_affinity = os.sched_getaffinity(0)
  numa = bind_to_gpu_numa_node(local)
  if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

  p = model_params()
  w = weights_lib.init_weights(p, seed=1)
  B, L, R = args.batch, p.max_length, p.total_rows
  cal = calibration_lib.parse_calibration_string(CALIBRATION)
  model = engine_lib.B200Model(p, w, max_batch=B, device=local, calibration=cal)

  # ---- inputs: NBUF distinct batches rotate so a step's rows are never L2-resident
  NBUF = 4
  row_bytes = B * R * L * 4
  host_rows = [synthetic.make_rows(p, B, seed=20240921 + 1 + rank * NBUF + i)[..., 0] for i in range(NBUF)]
  dev_rows = [model.alloc_device(row_bytes) for _ in range(NBUF)]
  for d, h in zip(dev_rows, host_rows):
    model.memcpy_h2d(d, h)
  dev_bases, dev_quals = model.alloc_device(B * L), model.alloc_device(B * L)
  dev_packed = []     # filled below once the packed form exists
  pin_addr, pin = [], []
  for h in host_rows:
    a, arr = engine_lib.alloc_pinned(row_bytes)
    arr.view(np.float32)[:] = h.reshape(-1)
    pin_addr.append(a)
    pin.append(arr)
  # packed form of the same batches (include/dcb200.h "packed input rows": what a producer of rows hands over)
  stride = model.packed_window_bytes
  packed_bytes = B * stride
  ppin_addr, ppin = [], []
  for h in host_rows:
    a, arr = engine_lib.alloc_pinned(packed_bytes)
    model.pack_rows(h, out=arr.reshape(B, stride))
    ppin_addr.append(a)
    ppin.append(arr)
  NPK = max(NBUF, int(140e6 // packed_bytes) + 1)     # resident packed batches rotate over > 126 MB (L2) of addresses
  for i in range(NPK):
    d = model.alloc_device(packed_bytes)
    model.memcpy_h2d(d, ppin[i % NBUF][:packed_bytes])
    dev_packed.append(d)
  out_addr, out_pin = engine_lib.alloc_pinned(2 * B * L)
  out_addr2, out_pin2 = engine_lib.alloc_pinned(2 * B * L)
  outs = (out_addr, out_addr2)
  FL = engine_lib.DCB_ROWS_ON_DEVICE | engine_lib.DCB_OUT_ON_DEVICE

  def step_resident(i):
    model.forward_raw(dev_rows[i % NBUF], B, FL, dev_bases, dev_quals)

  def step_e2e(i):
    model.forward_raw(pin_addr[i % NBUF], B, 0, out_addr, out_addr + B * L)

  def run_resident_pipelined(steps, packed=True):
    # same submission pattern with the rows already in HBM and device-side outputs: no host<->device traffic at all.
    # packed=True: the engine's packed row format (7.3 KB/window, include/dcb200.h); False: float32 [B,R,L] rows
    pending = None
    for i in range(steps):
      if packed:
        t = model.submit_packed_raw(dev_packed[i % NPK], B, FL, dev_bases, dev_quals)
      else:
        t = model.submit_raw(dev_rows[i % NBUF], B, FL, dev_bases, dev_quals)
      if pending is not None:
        model.wait_raw(pending)
        run_resident_pipelined.dev_ms += model.last_forward_ms()
      pending = t
    model.wait_raw(pending)
    run_resident_pipelined.dev_ms += model.last_forward_ms()
  run_resident_pipelined.dev_ms = 0.0

  def run_e2e_pipelined(steps, packed=True):
    # the call sequence of inference.run_model_on_examples: submit batch i, then collect batch i-1; every step's rows
    # go host->device (packed rows: dcb_submit_packed; float32 rows: dcb_submit) and every step's bases/quals come back
    # to the host inside the timed region
    pending = None
    for i in range(steps):
      if packed:
        t = model.submit_packed_raw(ppin_addr[i % NBUF], B, 0, outs[i % 2], outs[i % 2] + B * L)
      else:
        t = model.submit_raw(pin_addr[i % NBUF], B, 0, outs[i % 2], outs[i % 2] + B * L)
      if pending is not None:
        model.wait_raw(pending)
        run_resident_pipelined.dev_ms += model.last_forward_ms()
      pending = t
    model.wait_raw(pending)
    run_resident_pipelined.dev_ms += model.last_forward_ms()

  def barrier():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def timed(fn, steps):
    barrier()
    t0 = time.perf_counter()
    dev_ms = 0.0
    for i in range(steps):
      fn(i)
      dev_ms += model.last_forward_ms()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
      t = torch.tensor([dt, dev_ms], device="cuda", dtype=torch.float64)
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      dt, dev_ms = float(t[0]), float(t[1])
    barrier()
    return dt, dev_ms

  def reduce_max(*vals):
    if world == 1:
      return vals
    t = torch.tensor(list(vals), device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return tuple(float(x) for x in t)

  def trial(fn):
    """EXACTLY args.steps steps, bracketed by barrier + synchronize on both sides; wall time and summed device time,
    MAX over ranks."""
    run_resident_pipelined.dev_ms = 0.0
    barrier()
    t0 = time.perf_counter()
    fn(args.steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    dt, dev = reduce_max(dt, run_resident_pipelined.dev_ms)
    barrier()
    return dt, dev

  TRIALS = 5
  for i in range(args.warmup):
    step_resident(i)
  sampler = ClockSampler(local)
  sampler.start()
  # per-kernel device times right after warm-up, before the timed trials heat the GPU into its power cap: the state the
  # burst cuBLAS peak was measured in (reported next to the post-trial measurement, which is the `roofline` proper)
  model.set_profile(True)
  barrier()
  run_resident_pipelined(args.steps)
  torch.cuda.synchronize()
  prof_cool = model.get_profile()
  model.set_profile(False)
  run_e2e_pipelined(3)
  res_trials, e2e_trials = [], []
  for _ in range(TRIALS):       # resident and host-buffer trials alternate, so both see the same thermal / power state
    res_trials.append(trial(run_resident_pipelined))                             # per-kernel events OFF
    e2e_trials.append(trial(run_e2e_pipelined))
  if args.dump_outputs and rank == 0:
    # the host-buffer trials write elsewhere, so the device outputs still hold the last step of the last `value` trial
    bases, quals = np.empty((B, L), np.uint8), np.empty((B, L), np.uint8)
    model.memcpy_d2h(bases, dev_bases)
    model.memcpy_d2h(quals, dev_quals)
    dump_outputs(args.dump_outputs, bases=bases, quals=quals)
  res_f32 = [trial(lambda n: run_resident_pipelined(n, packed=False)) for _ in range(3)]
  run_e2e_pipelined(3, packed=False)
  f32_trials = [trial(lambda n: run_e2e_pipelined(n, packed=False)) for _ in range(3)]
  dt_e2e_f32 = sorted(t[0] for t in f32_trials)[1]
  for i in range(3):
    step_e2e(i)
  dt_e2e_blocking, _ = timed(step_e2e, args.steps)
  sampler.stop_flag.set()
  sampler.join(timeout=2)
  med = sorted(range(TRIALS), key=lambda i: res_trials[i][0])[TRIALS // 2]
  dt, dev_ms = res_trials[med]
  med_e = sorted(range(TRIALS), key=lambda i: e2e_trials[i][0])[TRIALS // 2]
  dt_e2e, dev_ms_e2e = e2e_trials[med_e]
  launches = model.last_forward_launches() * args.steps

  # ---- per-kernel device times (CUDA events around every launch on the engine's stream): a separate pass of the
  # same K steps, so the events do not sit inside the `value` trials
  model.set_profile(True)
  barrier()
  run_resident_pipelined(args.steps)
  torch.cuda.synchronize()
  prof = model.get_profile()
  model.set_profile(False)

  # ---- sustained: >= 2 s of back-to-back steps, kernel events on, own clock samples
  sus = None
  if rank == 0 or world > 1:
    n_sus = max(args.steps, int(2.2 / max(dt / args.steps, 1e-6)))
    sus_sampler = ClockSampler(local)
    sus_sampler.start()
    model.set_profile(True)
    barrier()
    t0 = time.perf_counter()
    run_resident_pipelined(n_sus)
    torch.cuda.synchronize()
    sus_dt = time.perf_counter() - t0
    sus_prof = model.get_profile()
    model.set_profile(False)
    sus_sampler.stop_flag.set()
    sus_sampler.join(timeout=2)
    (sus_dt,) = reduce_max(sus_dt)
    sus = dict(steps=n_sus, seconds=sus_dt, value=B * world * n_sus / sus_dt, prof=sus_prof, clocks=sus_sampler.summary())

  # ---- parity of what was just timed: the default path against the strict-fp32 path on the whole batch (device)
  par = None
  if rank == 0:
    from deepconsensus_b200 import parity as parity_lib
    fast = model.forward(host_rows[0], want_logits=True)
    strict = model.forward(host_rows[0], want_logits=True, strict=True)
    par = parity_lib.summary(parity_lib.compare(fast, strict, margin=0.25))
    par["of"] = ("default bf16 tensor-core path vs the engine's strict-fp32 path (reference arithmetic; pinned to the "
                 "oracle / reference-code goldens in tests/), all %d windows of one batch, on the device" % B)
    par["strict_ms_per_batch"] = model.last_ms

  # ---- BASELINE configs[3]: the same step fed by ONE reader rank over NCCL (grouped send/recv of packed chunks,
  # double-buffered; results gathered back) instead of every rank holding its own shard.  Secondary record: the
  # natural split for this path is the replica form above (no data-path collective).
  # Opt-in (--nccl-scatter): of three 8-GPU runs of this record one ended in an unexplained "unspecified launch failure" on
  # one receiving rank (not reproduced in 3000 overlapped steps on 2 GPUs, scripts/gpu_scatter_stress.py; DESIGN.md section 7),
  # and a secondary record must not be able to take the primary line down with it.
  scatter_info = None
  if world > 1 and args.nccl_scatter:
    from deepconsensus_b200 import parallel as parallel_lib
    feeder = parallel_lib.ScatterFeeder(packed_bytes, 2 * B * L, reader=0, device=torch.device("cuda", local))
    step_rows = None
    if rank == 0:
      one = torch.from_numpy(np.stack([ppin[i % NBUF][:packed_bytes] for i in range(2)])).to(feeder.device)   # 2 distinct steps
      step_rows = [one[i].unsqueeze(0).expand(world, packed_bytes).contiguous() for i in range(2)]
    res_ptr = feeder.results.data_ptr()

    def run_scatter(steps):
      feeder.scatter(0, step_rows[0] if rank == 0 else None)
      for i in range(steps):
        feeder.wait()                                             # chunk i landed (and results i-1 gathered)
        if i + 1 < steps:
          feeder.scatter((i + 1) & 1, step_rows[(i + 1) & 1] if rank == 0 else None)   # overlaps the kernels of step i
        t = model.submit_packed_raw(feeder.inbox[i & 1].data_ptr(), B, FL, res_ptr, res_ptr + B * L)
        model.wait_raw(t)
        feeder.gather()
      feeder.wait()
    run_scatter(3)
    sc_trials = [trial(run_scatter) for _ in range(3)]
    dt_sc = sorted(t[0] for t in sc_trials)[1]
    scatter_info = dict(value=B * world * args.steps / dt_sc, unit=UNIT, ms_per_step=dt_sc / args.steps * 1e3,
                        bytes_scattered_per_step=packed_bytes * (world - 1), bytes_gathered_per_step=2 * B * L * (world - 1),
                        call="rank 0 -> every rank: batch_isend_irecv (ncclGroupStart/Send/Recv/End) of packed chunks, "
                             "double-buffered; dcb_submit_packed on the received device buffer; results gathered on rank 0",
                        trials=[round(B * world * args.steps / t[0], 1) for t in sc_trials])

  # ---- the "next" row after the model path: per-read stitching of the outputs on the device (dcb_stitch), timed on
  # the device buffers the last forward wrote (128 reads of 8 windows), call-to-return including its own sync
  zs = np.arange(0, B + 1, 8, dtype=np.int32)
  if zs[-1] != B:
    zs = np.append(zs, B).astype(np.int32)
  st_seq, st_qual, st_len = model.alloc_device(B * L), model.alloc_device(B * L), model.alloc_device(4 * len(zs))
  for _ in range(3):
    model.stitch_raw(dev_bases, dev_quals, B, zs, FL, st_seq, st_qual, st_len)
  t0 = time.perf_counter()
  n_st = 50
  for _ in range(n_st):
    model.stitch_raw(dev_bases, dev_quals, B, zs, FL, st_seq, st_qual, st_len)
  stitch_us = (time.perf_counter() - t0) / n_st * 1e6
  stitch_info = dict(us_per_batch=stitch_us, windows=B, reads=int(len(zs) - 1), bytes_in=2 * B * L,
                     achieved_gbps=4 * B * L / (stitch_us * 1e-6) / 1e9,
                     note="get_full_sequence + remove_gaps for the whole batch; at 0.5 MB per batch the call is launch / "
                          "synchronisation latency, not HBM bandwidth")
  for d in (st_seq, st_qual, st_len):
    model.free_device(d)

  total_windows = B * world * args.steps
  value = total_windows / dt
  e2e_value = total_windows / dt_e2e
  F = flops_per_window(p)
  peaks = measured_peaks()
  # dominant kernel.  fused_oproj == 2: the whole encoder stack runs in ONE kernel (stack_pair_kernel) -- algorithmic
  # FLOPs per launch = tokens * layers * (8 d^2 + 4 d ff) + banded attention pairs; otherwise the per-layer fused
  # out-proj + FFN kernel: tokens * (4 d ff [+ 2 d d]).
  d, ff, wdw, Lp = p.hidden_size, p.filter_size, p.attn_win_size, p.max_length
  if prof["fused_oproj"] == 2:
    pairs = Lp * (2 * wdw + 1) - wdw * (wdw + 1)
    per_token = p.num_hidden_layers * (8.0 * d * d + 4.0 * d * ff + 4.0 * pairs * d / Lp)
    kname = ("stack_pair_kernel (all %d layers: QKV + banded attention + out-proj + FFN, residual in TMEM; final LayerNorm, fc1 "
             "and the quality epilogue in its tail -- their flops are not counted)" % p.num_hidden_layers)
  else:
    per_token = 4.0 * d * ff + (2.0 * d * d if prof["fused_oproj"] else 0.0)
    kname = "ffn_pair_kernel<fused out-proj>" if prof["fused_oproj"] else "ffn_pair_kernel"

  def kernel_tflops(pr):
    return pr["ffn_tokens"] * per_token / (pr["ffn_ms_total"] * 1e-3) / 1e12 if pr["ffn_ms_total"] > 0 else None
  ffn_tflops = kernel_tflops(prof)
  traffic = None
  tpath = os.path.join(ROOT, "profiles", "stack_dram_traffic.json" if prof["fused_oproj"] == 2 else "ffn_dram_traffic.json")
  if os.path.exists(tpath):
    with open(tpath) as f:
      traffic = json.load(f).get("dram_bytes_per_launch")
  kshare = {k: round(v["ms"] / max(sum(x["ms"] for x in prof["kernels"].values()), 1e-9), 4) for k, v in prof["kernels"].items()}
  peak_used, peak_src = peaks["bf16_tflops"], peaks["source"] + " (burst cuBLAS bf16; the K-step region is tens of ms)"
  roof = dict(bound="tensor", kernel=kname,
              achieved=ffn_tflops, flops_per_token=per_token, kernel_time_share=kshare,
              kernel_ms_per_step={k: round(v["ms"] / args.steps, 4) for k, v in prof["kernels"].items()}, peak=peak_used,
              unit="TFLOP/s", frac=(ffn_tflops / peak_used) if ffn_tflops else None,
              traffic=traffic, peak_source=peak_src,
              launches_timed=prof["ffn_launches"],
              avg_launch_ms=prof["ffn_ms_total"] / max(prof["ffn_launches"], 1),
              model_tflops_whole_step=value / world * F / 1e12,
              model_frac_of_peak=value / world * F / 1e12 / peak_used)
  cool = kernel_tflops(prof_cool)
  roof["first_pass_after_warmup"] = dict(achieved=cool, frac=(cool / peak_used) if cool else None,
                                         avg_launch_ms=prof_cool["ffn_ms_total"] / max(prof_cool["ffn_launches"], 1),
                                         note="same K steps timed before the trials (GPU not yet at its power cap, as when the "
                                              "burst peak was measured); `achieved` / `frac` above are from the pass after the trials")
  if sus is not None and peaks.get("bf16_tflops_sustained"):
    st = kernel_tflops(sus["prof"])
    roof["sustained"] = dict(seconds=round(sus["seconds"], 3), steps=sus["steps"], value=sus["value"],
                             achieved=st, peak=peaks["bf16_tflops_sustained"],
                             frac=(st / peaks["bf16_tflops_sustained"]) if st else None,
                             model_tflops_whole_step=sus["value"] / world * F / 1e12,
                             clocks=sus["clocks"],
                             note=">= 2 s of back-to-back steps (per-kernel events on); peak = sustained cuBLAS bf16")
  line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
              ms_per_step=dt / args.steps * 1e3, device_ms_per_step=dev_ms / args.steps,
              higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
              data="synthetic",
              config=config_dict(world, B),
              resident_float32_rows=dict(value=total_windows / sorted(t[0] for t in res_f32)[1],
                                         note="same region with float32 [B,R,L] rows resident instead of packed rows"),
              timing=dict(trials=TRIALS, reported="median trial; every trial = exactly %d steps between barrier+sync; value and "
                                                  "e2e trials alternate (same thermal / power state)" % args.steps,
                          value_trials=[round(total_windows / t[0], 1) for t in res_trials],
                          e2e_trials=[round(total_windows / t[0], 1) for t in e2e_trials],
                          l2="inputs rotate over %d resident packed batches (%.0f MB of addresses > 126 MB L2); every step also "
                             "streams the 151 MB fp32 residual image through L2" % (NPK, NPK * packed_bytes / 1e6),
                          input="packed rows, %d B/window (include/dcb200.h), resident in HBM" % stride,
                          gflop_per_window=F / 1e9),
              e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=packed_bytes * world,
                       d2h_bytes_per_step=2 * B * L * world, ms_per_step=dt_e2e / args.steps * 1e3,
                       device_ms_per_step=dev_ms_e2e / args.steps,
                       call="dcb_submit_packed/dcb_wait from pinned host memory, 2 batches in flight (as "
                            "inference.run_model_on_examples); input = packed rows, %d B/window "
                            "(include/dcb200.h), results = base + quality characters back on the host" % stride,
                       float32_rows=dict(value=total_windows / dt_e2e_f32, h2d_bytes_per_step=row_bytes * world,
                                         call="dcb_submit/dcb_wait on the reference's float32 [B,R,L] rows (%d B/window)"
                                              % (row_bytes // B)),
                       blocking_value=total_windows / dt_e2e_blocking,
                       blocking_call="dcb_forward on float32 rows, one batch at a time"),
              gpu_launches=launches, roofline=roof, parity=par, nccl_scatter=scatter_info, clocks=sampler.summary(), numa_node=numa, stitch=stitch_info)
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    os.sched_setaffinity(0, full_affinity)   # the CPU arm may use every host core again
    cores = cpu_threads()
    v, secs = cpu_reference_windows_per_sec(p, w, sample_windows=B, reps=2, threads=cores)
    line["cpu_baseline"] = dict(value=v, unit=UNIT, cores=cores, kind="port",
                                sample="the full batch of %d synthetic windows, 1 warm-up + 2 timed passes, torch-CPU fp32 "
                                       "oracle incl. argmax / QV (%.1f s/pass)" % (B, secs))
  if rank == 0:
    print(json.dumps(line))
  for d in dev_rows + dev_packed + [dev_bases, dev_quals]:
    model.free_device(d)
  for a in pin_addr + ppin_addr + [out_addr, out_addr2]:
    engine_lib.free_pinned(a)
  model.close()
  if world > 1:
    dist.destroy_process_group()


if __name__ == "__main__":
  main()
