#!/usr/bin/env python
"""Benchmark of the hot path: input samples/s through the 64-channel gammatone ERB bank.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--strategy slaney]
                  [--sharding streams|channels] [--distribute] [--dump-outputs DIR]

* A STEP is one pass of the bank over one resident batch of synthetic float32 streams:
  per GPU 4096 streams x 16384 samples (BASELINE.json config 4: "64-channel gammatone ERB
  bank x 4096 independent input streams, 1 GPU HBM-bound"); with N GPUs every rank owns its
  own 4096 streams (stream sharding, weak scaling; 8 ranks move the same 5.4e8 input samples
  per step as config 5's 65536 x 8192, whose own per-GPU shape is the ``cfg5`` record).
* ``value`` = input stream-samples/s of the whole job, device-timed with CUDA events on the
  launching stream, exactly K steps between barrier + synchronize, max over ranks.
* ``e2e`` = the same metric through the C-ABI host entry (``alz_apply_f32_host``) with PINNED
  HOST buffers: host->device copy of x and device->host copy of every output row inside the
  timed region, every step.
* ``roofline`` = algorithmic HBM bytes (260 B per input sample: 4 read + 64 x 4 written) over
  the measured launch duration, against the measured copy peak of MEASURED_PEAKS.json; ``burst``
  is the K-step region, ``sustained`` >= 2 s of back-to-back launches with its own clock record.
* ``--sharding channels`` (N > 1): the north-star shape -- rank 0 owns the input block, NCCL
  broadcast on a side stream overlapped with the previous block's kernel, every rank filters
  its slice of the 64 channels, outputs stay sharded; the in-place all-gather of the outputs is
  timed separately against the NVLink rate. ``--distribute`` (stream sharding): the batch starts
  on rank 0 and is scattered inside the timed region.
* ``cpu_baseline`` (rank 0, N = 1) and ``--impl reference``: the CPU restatement of the
  reference's evaluator (oracle/, kind "port": the reference itself is pure Python) on the host
  threads this process may use, median of 5 repetitions (``--impl reference``: K) on ONE bounded
  sample of the same workload.
* ``--dump-outputs DIR`` (GPU run, stream sharding): after the K timed steps, rank 0 writes
  ``DIR/y.npy``, float32 [n][64][T]: what the last timed step wrote to y[S][64][T] for a fixed,
  seeded sample of n streams (at most 32 MB; see ``output_sample``).  The inputs are seeded, so
  two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "samples/sec through 64-ch gammatone bank"
UNIT = "input-samples/s"
S_PER_GPU, T, C, RATE = 4096, 16384, 64, 48000
BYTES_PER_IN_SAMPLE = 4 + 4 * C     # SURVEY.md section 8(d)
NVLINK_GBS = 900.0                  # one direction of NVLink 5 per GPU (B200_PROFILING.md)
DUMP_BYTES = 32 << 20               # --dump-outputs: bytes of y written at most


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--strategy", default="slaney", choices=["slaney", "klapuri", "sampled"])
  ap.add_argument("--streams", type=int, default=S_PER_GPU, help="streams per GPU")
  ap.add_argument("--samples", type=int, default=T, help="samples per stream per step")
  ap.add_argument("--sharding", default="streams", choices=["streams", "channels"])
  ap.add_argument("--distribute", action="store_true", help="stream sharding: scatter the batch from rank 0 inside the timed region")
  ap.add_argument("--sustain-s", type=float, default=2.0, help="length of the sustained roofline run")
  ap.add_argument("--no-e2e", action="store_true")
  ap.add_argument("--no-cpu", action="store_true")
  ap.add_argument("--no-extras", action="store_true", help="skip the secondary records (strategies, cfg2/3/5, generic, stream API)")
  ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs as DIR/y.npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be >= 1")
  if args.dump_outputs and args.impl == "reference":
    ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
  return args


def peaks():
  try:
    with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
      return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
  except Exception:
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
  """DRAM bytes per launch of the headline kernel from the committed ncu capture."""
  try:
    with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as fh:
      return json.load(fh).get("dram_bytes_per_launch")
  except Exception:
    return None


def host_cpus():
  """Threads this process may really use: scheduler affinity, capped by the cgroup CPU quota."""
  try:
    n = len(os.sched_getaffinity(0))
  except Exception:
    n = os.cpu_count() or 1
  info = {"affinity": n, "cpu_count": os.cpu_count()}
  quota = None
  for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
    try:
      txt = open(path).read().split()
      if path.endswith("cpu.max"):
        if txt[0] != "max":
          quota = float(txt[0]) / float(txt[1])
      else:
        q = float(txt[0])
        if q > 0:
          quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
      break
    except Exception:
      continue
  info["cgroup_quota_cpus"] = quota
  threads = max(1, min(n, int(quota) if quota and quota >= 1 else n))
  try:
    info["loadavg_1m"] = os.getloadavg()[0]
  except Exception:
    pass
  return threads, info


class ClockSampler(object):
  """Samples SM clock / throttle reasons of one GPU during a timed region (NVML)."""

  def __init__(self, index):
    self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
    self._stop = threading.Event()
    self._thread = None
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nv = pynvml
      self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
    except Exception:
      self.nv = None

  def _run(self):
    nv = self.nv
    names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
             nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
             nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
             nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
             nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
    while not self._stop.is_set():
      try:
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for bit, name in names.items():
          if mask & bit:
            self.reasons.add(name)
        self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
      except Exception:
        pass
      self._stop.wait(0.004)

  def start(self):
    if self.nv is not None:
      self._thread = threading.Thread(target=self._run, daemon=True)
      self._thread.start()
    return self

  def stop(self):
    self._stop.set()
    if self._thread is not None:
      self._thread.join()
    s = sorted(self.samples)
    return {"sm_mhz": s[len(s) // 2] if s else None, "sm_min_mhz": s[0] if s else None, "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons), "samples": len(s), "power_w_max": max(self.power) if self.power else None}


def bank_sections(strategy):
  import audiolazy_b200 as ab
  return ab.gammatone_bank(rate=RATE, strategy=strategy)


# ------------------------------------------------------------------------------------------
# CPU legs (the only places bench.py touches oracle/)
# ------------------------------------------------------------------------------------------
class CpuPort(object):
  """The oracle (C restatement of the reference's evaluator) on `threads` host threads over ONE
  fixed sample of the bench workload, sized once so that a repetition takes about `rep_s`."""

  def __init__(self, bank, threads, rep_s=1.5, t_cpu=2048):
    import numpy as np
    import oracle
    self.oracle, self.np = oracle, np
    self.sections = bank.sections()
    self.threads, self.t_cpu = threads, t_cpu
    rng = np.random.default_rng(0)
    per_thread = 4                       # streams per thread in the sizing probe: thread start-up must not dominate
    probe = rng.uniform(-1, 1, (threads * per_thread, t_cpu)).astype(np.float32)
    out = np.zeros((probe.shape[0], C, t_cpu), dtype=np.float32)   # zeros: pages touched before the clock starts
    oracle.bank_apply_f32(probe, self.sections, threads=threads, out=out)     # untimed: library load, thread pool warm-up
    t0 = time.perf_counter()
    oracle.bank_apply_f32(probe, self.sections, threads=threads, out=out)
    rate = probe.shape[0] * t_cpu / (time.perf_counter() - t0)
    n = int(max(threads, min(S_PER_GPU, (rate * rep_s / t_cpu) // threads * threads)))
    self.x = rng.uniform(-1, 1, (n, t_cpu)).astype(np.float32)
    self.out = np.zeros((n, C, t_cpu), dtype=np.float32)
    self.sample = "%d streams x %d samples x %d channels, %d threads" % (n, t_cpu, C, threads)

  def once(self):
    t0 = time.perf_counter()
    self.oracle.bank_apply_f32(self.x, self.sections, threads=self.threads, out=self.out)
    return self.x.size / (time.perf_counter() - t0)

  def measure(self, reps, warm=1):
    for _ in range(warm):
      self.once()
    vals = [self.once() for _ in range(max(1, reps))]
    return {"value": statistics.median(vals), "min": min(vals), "max": max(vals), "reps": len(vals)}


def python_exec_throughput(bank, n=3000):
  """CPython cost of the reference's own evaluation strategy -- per-section generator functions
  generated as source and exec'ed, nested lazily (oracle.py_compiled_cascade) -- for the 64-channel
  bank on one core: in-samples/s (8 of the 64 channels timed, x8)."""
  import numpy as np
  import oracle
  sections = bank.sections()
  x = np.random.default_rng(0).uniform(-1, 1, n).astype(np.float32).astype(float).tolist()
  t0 = time.perf_counter()
  for ch in sections[::8]:
    list(oracle.py_compiled_cascade(ch, x))
  return len(x) / ((time.perf_counter() - t0) * 8)


def run_reference(args):
  """--impl reference: the CPU port on the usable host threads; rank 0 only."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  threads, cpu_info = host_cpus()
  bank = bank_sections(args.strategy)
  port = CpuPort(bank, threads)
  m = port.measure(args.steps, warm=max(args.warmup, 1))
  value = m["value"]
  line = {
    "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
    "warmup": args.warmup, "ms_per_step": args.streams * args.samples / value * 1e3, "higher_is_better": True,
    "scaling": "weak", "vs_baseline": None,
    "dtype": "f64", "data": "synthetic",
    "config": {"workload": "64-ch gammatone ERB bank (%s), fs 48 kHz, CPU port of the reference evaluator on a "
                           "bounded sample of the %d x %d stream batch" % (args.strategy, args.streams, args.samples),
               "ms_per_step_note": "extrapolated from the sample to the whole batch (streams are independent: the "
                                   "cost is linear in their number)",
               "value_note": "median of %d repetitions on one fixed sample" % m["reps"]},
    "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": port.sample,
                     "min": m["min"], "max": m["max"], "reps": m["reps"], "host": cpu_info},
    "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    "gpu_launches": 0,
  }
  print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------
class Timer(object):
  """Device timing of `fn` repeated n times on torch's current stream (where the library launches)."""

  def __init__(self, torch, dev, barrier):
    self.torch, self.dev, self.barrier = torch, dev, barrier

  def run(self, fn, n):
    torch = self.torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    self.barrier()
    e0.record()
    for _ in range(n):
      fn()
    e1.record()
    self.barrier()
    return e0.elapsed_time(e1)


def output_sample(y):
  """A fixed, seeded sample of the [S][C][T] float32 device tensor y, as a host array of at most
  DUMP_BYTES: whole streams (every channel and sample) chosen by numpy default_rng(0), and when one
  stream alone is larger than that, a sorted seeded sample of its time positions too."""
  import numpy as np
  import torch
  S, Cn, Tn = y.shape
  rng = np.random.default_rng(0)
  row_bytes = Cn * Tn * y.element_size()
  streams = np.sort(rng.choice(S, int(min(S, max(1, DUMP_BYTES // row_bytes))), replace=False))
  out = y[torch.as_tensor(streams, device=y.device)]
  if len(streams) * row_bytes > DUMP_BYTES:
    times = np.sort(rng.choice(Tn, int(DUMP_BYTES // (Cn * y.element_size())), replace=False))
    out = out[:, :, torch.as_tensor(times, device=y.device)]
  return out.cpu().numpy()


def device_record(torch, dev, plan, S, Tn, steps=5, warm=2, flush=None):
  """ms per launch of one plan over a resident [S][Tn] batch (best-effort secondary record)."""
  Cn = plan.n_channels
  x = torch.rand((S, Tn), device=dev) * 2 - 1
  y = torch.empty((S, Cn, Tn), dtype=torch.float32, device=dev)
  st = torch.zeros(max(1, plan.state_doubles(S)), dtype=torch.float64, device=dev)
  cur = torch.cuda.current_stream(dev).cuda_stream
  for _ in range(warm):
    plan.apply(x.data_ptr(), y.data_ptr(), st.data_ptr(), S, Tn, Tn, Tn, cur)
  torch.cuda.synchronize(dev)
  times = []
  for _ in range(steps):
    if flush is not None:
      flush.zero_()                        # small cases fit in L2: evict between timed launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    plan.apply(x.data_ptr(), y.data_ptr(), st.data_ptr(), S, Tn, Tn, Tn, cur)
    e1.record()
    torch.cuda.synchronize(dev)
    times.append(e0.elapsed_time(e1))
  ms = statistics.median(times)
  del x, y, st
  return {"ms": ms, "input_samples_per_s": S * Tn / (ms * 1e-3), "gbs": (4 + 4 * Cn) * S * Tn / (ms * 1e-3) / 1e9,
          "streams": S, "samples": Tn, "channels": Cn}


def extras(torch, dev, args, peak):
  """Secondary records (rank 0, N = 1): the other strategies, cfg 2 / 3 / 5, the generic kernel, the Stream API."""
  import numpy as np
  import audiolazy_b200 as ab
  from audiolazy_b200 import _capi
  out = {}
  flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
  S, Tn = args.streams, args.samples
  try:
    strat = {}
    for name in ("slaney", "klapuri", "sampled"):
      if name == args.strategy:
        continue
      plan = bank_sections(name).device_bank().plan
      r = device_record(torch, dev, plan, S, Tn)
      r["roofline_frac"] = r["gbs"] / peak
      r["fp32_tier_channels"] = plan.n_fp32_channels
      strat[name] = r
    out["strategies"] = strat
  except Exception as exc:                                            # a secondary record must never kill the headline
    out["strategies"] = {"error": repr(exc)}
  try:
    # the same bank writing y[C][S][T] (alz_apply_f32_ex): a warp's 32 output rows are 64 KB apart instead of 4 MB
    plan = bank_sections(args.strategy).device_bank().plan
    xx = torch.rand((S, Tn), device=dev) * 2 - 1
    yy = torch.empty((C, S, Tn), dtype=torch.float32, device=dev)
    st = torch.zeros(plan.state_doubles(S), dtype=torch.float64, device=dev)
    cur = torch.cuda.current_stream(dev).cuda_stream
    times = []
    for i in range(7):
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      plan.apply_ex(xx.data_ptr(), yy.data_ptr(), st.data_ptr(), S, Tn, Tn, S * Tn, Tn, cur)
      e1.record()
      torch.cuda.synchronize(dev)
      if i >= 2:
        times.append(e0.elapsed_time(e1))
    ms = statistics.median(times)
    gbs = BYTES_PER_IN_SAMPLE * S * Tn / (ms * 1e-3) / 1e9
    out["channel_major_layout"] = {"ms": ms, "input_samples_per_s": S * Tn / (ms * 1e-3), "gbs": gbs, "roofline_frac": gbs / peak,
                                   "note": "secondary: output written as y[C][S][T] instead of the headline's y[S][C][T]"}
    del xx, yy, st
  except Exception as exc:
    out["channel_major_layout"] = {"error": repr(exc)}
  try:
    import scipy.signal as sig
    sos = sig.butter(8, 0.25, output="sos")
    cfg2 = _capi.Plan([[(r[:3].tolist(), r[3:].tolist()) for r in sos]])
    out["cfg2"] = dict(device_record(torch, dev, cfg2, 1, 1000000, flush=flush),
                       workload="8th-order Butterworth lowpass as 4 biquads, 1 stream x 1e6 samples (time-parallel path)")
    out["cfg3"] = dict(device_record(torch, dev, bank_sections(args.strategy).device_bank().plan, 1, 1000000, flush=flush),
                       workload="64-ch bank, 1 stream x 1e6 samples (time-parallel path)")
    out["few_streams"] = {
      "16x1e6": device_record(torch, dev, bank_sections(args.strategy).device_bank().plan, 16, 1000000, steps=3, warm=1),
      "256x65536": device_record(torch, dev, bank_sections(args.strategy).device_bank().plan, 256, 65536, steps=3, warm=1)}
  except Exception as exc:
    out["cfg2"] = {"error": repr(exc)}
  try:
    out["cfg5"] = dict(device_record(torch, dev, bank_sections(args.strategy).device_bank().plan, 8192, 8192),
                       workload="BASELINE config 5 per-GPU shape: 8192 streams x 8192 samples")
    out["cfg5"]["roofline_frac"] = out["cfg5"]["gbs"] / peak
  except Exception as exc:
    out["cfg5"] = {"error": repr(exc)}
  try:
    gen = {}
    comb = ab.comb.fb(37, .8)
    plan = _capi.Plan([comb.sections()])
    gen["comb_fb_37_0.8"] = device_record(torch, dev, plan, S * 16, Tn, steps=3, warm=1)
    rng = np.random.default_rng(5)
    lpc_a = [1.0] + (rng.uniform(-1, 1, 12) * 0.5 ** np.arange(1, 13)).tolist()
    gen["lpc12_analysis_fir"] = device_record(torch, dev, _capi.Plan([[(lpc_a, [1.0])]]), S * 16, Tn, steps=3, warm=1)
    gen["lpc12_synthesis_allpole"] = device_record(torch, dev, _capi.Plan([[([1.0], lpc_a)]]), S * 16, Tn, steps=3, warm=1)
    gen["biquad_kernel_reference"] = device_record(torch, dev, _capi.Plan([[([1.0, 0.5, 0.2], [1.0, -0.3, 0.1])]]), S * 16, Tn, steps=3, warm=1)
    gen["note"] = "single-channel plans over %d streams x %d samples (8 B per sample); kernels: window family (one section of " \
                  "any order / sparsity: dense near taps in registers, far taps prefetched from the state ring); " \
                  "biquad_kernel_reference = one float64 biquad on the biquad kernel at the same shape" % (S * 16, Tn)
    out["generic"] = gen
  except Exception as exc:
    out["generic"] = {"error": repr(exc)}
  try:
    import oracle
    api = {}
    x1 = np.random.default_rng(1).uniform(-1, 1, 48000).astype(np.float32).astype(float).tolist()
    f1 = ab.ZFilter([1, 7, 2], [1, 0.5, 0.2])
    list(f1(x1[:512]))
    t0 = time.perf_counter(); n1 = len(list(f1(x1))); t_ours = time.perf_counter() - t0
    t0 = time.perf_counter(); list(oracle.py_compiled_cascade([([1, 7, 2], [1, 0.5, 0.2])], x1)); t_ref = time.perf_counter() - t0
    api["cfg1"] = {"ours_samples_per_s": n1 / t_ours, "python_port_samples_per_s": n1 / t_ref, "samples": n1}
    x2 = np.random.default_rng(2).uniform(-1, 1, 1000000).astype(np.float32)
    casc = ab.CascadeFilter([ab.ZFilter(r[:3].tolist(), r[3:].tolist()) for r in sos])
    t0 = time.perf_counter(); n2 = len(list(casc(x2))); t_ours = time.perf_counter() - t0
    x2l = x2[:200000].astype(float).tolist()
    t0 = time.perf_counter()
    list(oracle.py_compiled_cascade([(r[:3].tolist(), r[3:].tolist()) for r in sos], x2l))
    t_ref = time.perf_counter() - t0
    api["cfg2"] = {"ours_samples_per_s": n2 / t_ours, "python_port_samples_per_s": len(x2l) / t_ref, "samples": n2}
    api["note"] = "list(filt(x)) wall time on one host core: the lazy Stream API of this package (block pump -> GPU -> " \
                  "Python floats) vs the exec-compiled pure-Python port of the reference's evaluator (oracle.py_compiled_cascade)"
    out["stream_api"] = api
  except Exception as exc:
    out["stream_api"] = {"error": repr(exc)}
  del flush
  return out


def run_ours(args):
  import numpy as np
  import torch
  import torch.distributed as dist
  from audiolazy_b200 import _capi

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if not torch.cuda.is_available():
    raise SystemExit("bench.py needs a GPU (there is no CPU fallback)")
  if args.dump_outputs and args.sharding == "channels" and world > 1:
    raise SystemExit("--dump-outputs is not supported with --sharding channels")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  distributed = world > 1
  if distributed:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version / debug lines must not mix with the JSON line on stdout
    try:                                                      # NCCL kernels on a high-priority stream: a broadcast issued under a
      opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)   # running bank kernel gets SM slots as soon as CTAs retire
      dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    except Exception:
      dist.init_process_group("nccl", device_id=dev)

  def barrier():
    if distributed:
      dist.barrier()
    torch.cuda.synchronize(dev)

  def max_over_ranks(v):
    t = torch.tensor([v], dtype=torch.float64, device=dev)
    if distributed:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  if args.sharding == "channels" and distributed:
    return run_channel_sharded(args, torch, dist, dev, world, rank, local, barrier, max_over_ranks)

  S, Tn = args.streams, args.samples
  bank = bank_sections(args.strategy)
  plan = bank.device_bank().plan
  tiers, _ = plan.tiers()
  gen = torch.Generator(device=dev)
  gen.manual_seed(1234 + rank)
  y = torch.empty((S, C, Tn), dtype=torch.float32, device=dev)
  state = torch.zeros(plan.state_doubles(S), dtype=torch.float64, device=dev)
  cur = torch.cuda.current_stream(dev).cuda_stream
  distribute = bool(args.distribute and distributed)
  if distribute:
    # the whole batch starts on rank 0; every step scatters it (NCCL) before the kernels run
    from audiolazy_b200.parallel import ShardedBank
    sb = ShardedBank(bank, mode="streams")
    x_full = (torch.rand((S * world, Tn), device=dev, generator=gen) * 2 - 1) if rank == 0 else None
    x = torch.empty((S, Tn), dtype=torch.float32, device=dev)

    def step():
      sb.scatter_input_into(x_full, x, src=0)
      plan.apply(x.data_ptr(), y.data_ptr(), state.data_ptr(), S, Tn, Tn, Tn, cur)
  else:
    x = torch.rand((S, Tn), device=dev, generator=gen) * 2 - 1          # synthetic uniform(-1, 1) float32

    def step():
      plan.apply(x.data_ptr(), y.data_ptr(), state.data_ptr(), S, Tn, Tn, Tn, cur)

  timer = Timer(torch, dev, barrier)
  for _ in range(max(args.warmup, 3)):
    step()
  barrier()
  sampler = ClockSampler(local).start()
  launches0 = _capi.launch_count()
  ms_total = max_over_ranks(timer.run(step, args.steps))
  launches = _capi.launch_count() - launches0
  clocks = sampler.stop()
  ms_per_step = ms_total / args.steps
  value = world * S * Tn / (ms_per_step * 1e-3)
  if args.dump_outputs and rank == 0:        # before anything below launches on y again
    os.makedirs(args.dump_outputs, exist_ok=True)
    np.save(os.path.join(args.dump_outputs, "y.npy"), output_sample(y))

  # ---- sustained: >= sustain_s of back-to-back launches, own clock record --------------------
  sustained = None
  if args.sustain_s > 0:
    n_sus = max(args.steps, int(args.sustain_s * 1e3 / ms_per_step) + 1)
    sampler = ClockSampler(local).start()
    ms_sus = max_over_ranks(timer.run(step, n_sus)) / n_sus
    sustained = {"ms_per_step": ms_sus, "steps": n_sus, "seconds": ms_sus * n_sus * 1e-3, "clocks": sampler.stop()}

  # ---- config 5's per-GPU shape (8192 x 8192), all ranks ---------------------------------------
  cfg5 = None
  if not args.no_extras and (S, Tn) == (S_PER_GPU, T):
    del x, y
    S5 = T5 = 8192
    x5 = torch.rand((S5, T5), device=dev, generator=gen) * 2 - 1
    y5 = torch.empty((S5, C, T5), dtype=torch.float32, device=dev)
    st5 = torch.zeros(plan.state_doubles(S5), dtype=torch.float64, device=dev)
    f5 = lambda: plan.apply(x5.data_ptr(), y5.data_ptr(), st5.data_ptr(), S5, T5, T5, T5, cur)
    for _ in range(3):
      f5()
    ms5 = max_over_ranks(timer.run(f5, 10)) / 10
    cfg5 = {"workload": "BASELINE config 5: 64-ch bank x %d streams x %d samples, %d per GPU" % (S5 * world, T5, S5),
            "ms_per_step": ms5, "value": world * S5 * T5 / (ms5 * 1e-3), "unit": UNIT,
            "gbs_per_gpu": BYTES_PER_IN_SAMPLE * S5 * T5 / (ms5 * 1e-3) / 1e9}
    del x5, y5, st5
    x = torch.rand((S, Tn), device=dev, generator=gen) * 2 - 1
    y = torch.empty((S, C, Tn), dtype=torch.float32, device=dev)

  # ---- end to end through the host-buffer C-ABI entry ------------------------------------
  e2e = None
  if not args.no_e2e:
    e2e = run_e2e(args, torch, dev, plan, x, world, barrier, max_over_ranks)

  def multi_gpu_records():
    """The batch scattered from rank 0; the channel-sharded north-star shape (all ranks take part)."""
    multi = {}
    torch.cuda.empty_cache()
    if not distribute:
      try:
        from audiolazy_b200.parallel import ShardedBank
        sbs = ShardedBank(bank, mode="streams")
        Sd = 1024
        xf = (torch.rand((Sd * world, Tn), device=dev, generator=gen) * 2 - 1) if rank == 0 else None
        xd = torch.empty((Sd, Tn), dtype=torch.float32, device=dev)
        yd = torch.empty((Sd, C, Tn), dtype=torch.float32, device=dev)
        std = torch.zeros(plan.state_doubles(Sd), dtype=torch.float64, device=dev)

        def step_d():
          sbs.scatter_input_into(xf, xd, src=0)
          plan.apply(xd.data_ptr(), yd.data_ptr(), std.data_ptr(), Sd, Tn, Tn, Tn, cur)

        def step_r():
          plan.apply(xd.data_ptr(), yd.data_ptr(), std.data_ptr(), Sd, Tn, Tn, Tn, cur)
        for _ in range(3):
          step_d()
        ms_d = max_over_ranks(timer.run(step_d, 10)) / 10
        ms_r = max_over_ranks(timer.run(step_r, 10)) / 10
        multi["distribute"] = {"workload": "stream sharding, %d streams x %d samples per GPU, the whole batch starts on rank 0 and "
                                           "is scattered by NCCL inside the timed region" % (Sd, Tn),
                               "value": world * Sd * Tn / (ms_d * 1e-3), "unit": UNIT, "ms_per_step": ms_d,
                               "ms_per_step_resident": ms_r, "scatter_overhead_frac": ms_d / ms_r - 1.0}
        del xf, xd, yd, std
      except Exception as exc:
        multi["distribute"] = {"error": repr(exc)}
    try:
      multi["channel_sharded"] = channel_sharded_record(args, torch, dist, dev, world, rank, local, barrier, max_over_ranks,
                                                        4096, 4096, 10)
    except Exception as exc:
      multi["channel_sharded"] = {"error": repr(exc)}
    return multi

  line = None
  if rank == 0:
    peak, peak_src = peaks()
    achieved = BYTES_PER_IN_SAMPLE * S * Tn / (ms_per_step * 1e-3) / 1e9          # per GPU, GB/s
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": ncu_traffic(), "peak_source": peak_src,
            "burst": {"achieved": achieved, "frac": achieved / peak, "seconds": ms_total * 1e-3},
            "kernel": "alz_biquad_tma_kernel<K=4,NB=2,MONIC=2>: %d of %d channels on the float32 tier (plan-time probe, "
                      "tolerance %.1e), the rest float64; DESIGN.md section 3" % (int(tiers.sum()), len(tiers), plan.tier_tol)}
    if sustained is not None:
      a_s = BYTES_PER_IN_SAMPLE * S * Tn / (sustained["ms_per_step"] * 1e-3) / 1e9
      roof["sustained"] = dict(sustained, achieved=a_s, frac=a_s / peak)
    line = {
      "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
      "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "f64", "data": "synthetic",
      "config": {"workload": "64-ch gammatone ERB bank (%s, 50 Hz-20 kHz ERB-rate spaced, fs 48 kHz) x %d streams x %d "
                             "samples per GPU (BASELINE config 4 per GPU)" % (args.strategy, S, Tn),
                 "streams_per_gpu": S, "samples_per_stream": Tn, "channels": C,
                 "sharding": "streams, batch scattered from rank 0 by NCCL inside the timed region" if distribute
                 else "streams (inputs resident per rank, no data-path collective)",
                 "io_dtype": "float32", "arithmetic": "float64 recurrence; float32 recurrence on the channels whose "
                 "plan-time probe error is <= %.1e (%d of %d)" % (plan.tier_tol, int(tiers.sum()), len(tiers)),
                 "l2": "inputs (%.0f MB) and outputs (%.1f GB) per step exceed the 126 MB L2"
                 % (S * Tn * 4 / 1e6, S * C * Tn * 4 / 1e9),
                 "realtime_48k_streams": value / RATE},
      "clocks": clocks, "gpu_launches": int(launches),
      "roofline": roof,
    }
    if e2e is not None:
      line["e2e"] = e2e
    if cfg5 is not None:
      line["cfg5"] = cfg5
    if world == 1 and not args.no_extras:
      line.update(extras(torch, dev, args, peak))
    if world == 1 and not args.no_cpu:
      threads, cpu_info = host_cpus()
      port = CpuPort(bank, threads)
      m = port.measure(5)
      line["cpu_baseline"] = {"value": m["value"], "unit": UNIT, "cores": threads, "kind": "port", "sample": port.sample,
                              "min": m["min"], "max": m["max"], "reps": m["reps"], "host": cpu_info,
                              "python_exec_1core": python_exec_throughput(bank)}
  if distributed and not args.no_extras:
    # The secondary multi-GPU records run AFTER the headline has been measured; a watchdog thread makes sure a hung
    # collective there cannot cost the line: after 300 s rank 0 prints what it has and every rank leaves.
    def bail():
      if rank == 0:
        line["multi_gpu_records"] = "timed out"
        print(json.dumps(line), flush=True)
      os._exit(0)
    dog = threading.Timer(300.0, bail)
    dog.daemon = True
    dog.start()
    del x, y
    multi = multi_gpu_records()
    dog.cancel()
    if rank == 0:
      line.update(multi)
  if rank == 0:
    print(json.dumps(line), flush=True)
  if distributed:
    dist.barrier()
    dist.destroy_process_group()


def run_e2e(args, torch, dev, plan, x, world, barrier, max_over_ranks):
  """Same metric through alz_apply_f32_host: pinned host buffers (allocated by the library on the GPU's
  NUMA node), H2D of x and D2H of every output row inside the timed region, every step."""
  from audiolazy_b200 import _capi
  S, Tn = args.streams, args.samples
  Se = S
  try:
    import psutil
    avail = psutil.virtual_memory().available
    per_stream = (C + 1) * Tn * 4
    Se = int(max(32, min(S, (avail * 0.4 / world) // per_stream // 32 * 32)))
  except Exception:
    pass
  xh = _capi.HostBuffer((Se, Tn))
  yh = _capi.HostBuffer((Se, C, Tn))
  xh.array[...] = x[:Se].cpu().numpy()
  state = torch.zeros(plan.state_doubles(Se), dtype=torch.float64, device=dev)
  torch.cuda.synchronize(dev)
  plan.apply_host(xh.array, yh.array, state.data_ptr())                  # warm-up: allocates the staging buffers
  k_e2e = max(1, min(args.steps, 3))
  barrier()
  t0 = time.perf_counter()
  for _ in range(k_e2e):
    plan.apply_host(xh.array, yh.array, state.data_ptr())                # H2D x, kernel, D2H y: all inside, synchronous
  torch.cuda.synchronize(dev)
  dt = max_over_ranks(time.perf_counter() - t0)
  h2d, d2h = Se * Tn * 4, Se * C * Tn * 4
  e2e = {"value": world * Se * Tn * k_e2e / dt, "unit": UNIT,
         "h2d_bytes_per_step": world * h2d, "d2h_bytes_per_step": world * d2h,
         "steps": k_e2e, "streams_per_gpu": Se, "pcie_gbs_per_gpu": (h2d + d2h) * k_e2e / dt / 1e9,
         "host_buffers": "pinned, numa node %s" % xh.numa_node,
         "note": "alz_apply_f32_host with pinned host buffers; PCIe-bound on the 256 B/sample output"}
  # second figure: the on-device envelope consumer shrinks the D2H stream by the decimation factor
  try:
    decim = 64
    eh = _capi.HostBuffer((Se, C, Tn // decim))
    env_kw = dict(decim=decim, mode="abs", g=1.0 - 0.99388, R=0.99388)      # envelope.abs with the reference's default cutoff pi / 512
    plan.apply_envelope_host(xh.array, eh.array, **env_kw)
    barrier()
    t0 = time.perf_counter()
    for _ in range(k_e2e):
      plan.apply_envelope_host(xh.array, eh.array, **env_kw)
    torch.cuda.synchronize(dev)
    dt2 = max_over_ranks(time.perf_counter() - t0)
    e2e["envelope_consumer"] = {
      "value": world * Se * Tn * k_e2e / dt2, "unit": UNIT, "decimation": decim,
      "d2h_bytes_per_step": world * Se * C * (Tn // decim) * 4,
      "note": "fused on-device |y| -> one-pole lowpass -> keep every %d-th sample (1 kHz envelope per channel), host "
              "buffers in and out; a DIFFERENT output than e2e.value's (labelled, not the headline)" % decim}
    eh.free()
  except Exception as exc:
    e2e["envelope_consumer"] = {"unavailable": repr(exc)}
  xh.free()
  yh.free()
  return e2e


def channel_sharded_record(args, torch, dist, dev, world, rank, local, barrier, max_over_ranks, S, Tn, steps):
  """North-star multi-GPU shape: channels sharded, the input block broadcast from rank 0 (NCCL, side stream,
  under the previous block's kernel), outputs stay sharded; gather (in-place all-gather, and the fused
  peer-memory store into rank 0) timed separately. Every rank takes part; the dict is meaningful on rank 0."""
  from audiolazy_b200 import _capi
  from audiolazy_b200.parallel import PeerOutput, ShardedBank
  bank = bank_sections(args.strategy)
  sb = ShardedBank(bank, mode="channels")
  Cl = sb.c_hi - sb.c_lo
  gen = torch.Generator(device=dev)
  gen.manual_seed(1234)
  # rank 0 owns the data; the other ranks' buffers are filled by the broadcasts only
  xb = [(torch.rand((S, Tn), device=dev, generator=gen) * 2 - 1) if rank == 0 else
        torch.zeros((S, Tn), dtype=torch.float32, device=dev) for _ in range(2)]
  y = sb.alloc_output(S, Tn)
  state = sb.local.new_state(S)
  timer = Timer(torch, dev, barrier)
  # first without an SM partition (the bank kernel's CTAs on every SM: NCCL's CTAs find no room until it ends) ...
  plain = sb.pipeline(xb, y, state)
  for _ in range(3):
    plain.step()
  plain.drain()
  ms_plain = max_over_ranks(timer.run(plain.step, steps)) / steps
  plain.drain()
  # ... then with the bank kernel confined to a green-context partition when it under-fills the machine anyway
  try:
    pipe = sb.pipeline(xb, y, state, compute_sms="auto")
  except Exception:
    pipe = plain
  for _ in range(3):
    pipe.step()
  pipe.drain()
  barrier()
  sampler = ClockSampler(local).start()
  launches0 = _capi.launch_count()
  ms = max_over_ranks(timer.run(pipe.step, steps)) / steps
  pipe.drain()
  launches = _capi.launch_count() - launches0
  clocks = sampler.stop()
  ms_nc = max_over_ranks(timer.run(lambda: pipe.compute_only(partition=True), steps)) / steps
  ms_bc = max_over_ranks(timer.run(lambda: sb.broadcast_input(xb[0], src=0), 10)) / 10
  rec = {"workload": "64-ch gammatone ERB bank (%s) x %d streams x %d samples per block, CHANNELS sharded over %d GPUs (%d "
                     "per GPU); input block broadcast from rank 0 by NCCL on a side stream under the previous block's "
                     "kernel; outputs stay sharded" % (args.strategy, S, Tn, world, Cl),
         "value": S * Tn / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "scaling": "strong",
         "gbs_per_gpu": (4 + 4 * Cl) * S * Tn / (ms * 1e-3) / 1e9, "clocks": clocks, "gpu_launches": int(launches),
         "collective": {"broadcast_ms": ms_bc, "broadcast_gbs": S * Tn * 4 / (ms_bc * 1e-3) / 1e9,
                        "step_ms_with_broadcast": ms, "step_ms_compute_only": ms_nc,
                        "overhead_frac": ms / ms_nc - 1.0, "broadcast_hidden": bool(ms <= 1.03 * ms_nc),
                        "compute_sms": pipe.partition.sm_count if pipe.partition is not None else None,
                        "step_ms_without_sm_partition": ms_plain,
                        "note": "the bank kernel runs on a green-context stream that owns compute_sms SMs (when it under-fills "
                                "the machine), so that NCCL's CTAs find free SMs while it runs"}}
  recv_bytes = S * (C - Cl) * Tn * 4          # what one rank ingests when it collects all channels
  try:
    gbuf = sb.alloc_gather(S, Tn)
    sb.gather_output_into(y, gbuf)
    ms_g = max_over_ranks(timer.run(lambda: sb.gather_output_into(y, gbuf), 3)) / 3
    rec["nvlink"] = {"gather_ms": ms_g, "recv_gbs_per_gpu": recv_bytes / (ms_g * 1e-3) / 1e9, "peak_gbs": NVLINK_GBS,
                     "frac": recv_bytes / (ms_g * 1e-3) / 1e9 / NVLINK_GBS,
                     "note": "ONE in-place all_gather_into_tensor of every rank's y[S][C/N][T] into [N][S][C/N][T] on every "
                             "rank; NOT on the throughput path (SURVEY.md section 8e): outputs stay sharded"}
    del gbuf
  except Exception as exc:
    rec["nvlink"] = {"error": repr(exc)}
  try:
    po = PeerOutput(S, C, Tn, dst=0)
    st2 = sb.local.new_state(S)

    def fused():
      sb.apply_into(xb[0], po, state=st2)
      po.fence()
    fused()
    ms_p = max_over_ranks(timer.run(fused, 3)) / 3
    rec["peer_store"] = {"ms": ms_p, "into_rank0_gbs": recv_bytes / (ms_p * 1e-3) / 1e9, "frac_of_nvlink": recv_bytes / (ms_p * 1e-3) / 1e9 / NVLINK_GBS,
                         "note": "fused compute + collective: every rank's kernel stores its channel rows (TMA) straight into rank 0's "
                                 "y[S][C][T] through NVLink peer memory (symmetric memory); no gather runs afterwards"}
    del po
  except Exception as exc:
    rec["peer_store"] = {"unavailable": repr(exc)}
  pipe.close()
  del xb, y, pipe, plain
  return rec


def run_channel_sharded(args, torch, dist, dev, world, rank, local, barrier, max_over_ranks):
  """--sharding channels: the channel-sharded record as the main line."""
  S, Tn = args.streams, args.samples
  rec = channel_sharded_record(args, torch, dist, dev, world, rank, local, barrier, max_over_ranks, S, Tn, args.steps)
  if rank == 0:
    peak, peak_src = peaks()
    line = {
      "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 3,
      "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
      "data": "synthetic",
      "config": {"workload": rec["workload"], "sharding": "channels", "streams": S, "samples_per_stream": Tn, "channels": C},
      "clocks": rec["clocks"], "gpu_launches": rec["gpu_launches"],
      "roofline": {"bound": "hbm", "achieved": rec["gbs_per_gpu"], "peak": peak, "unit": "GB/s", "frac": rec["gbs_per_gpu"] / peak,
                   "traffic": None, "peak_source": peak_src, "note": "per GPU: (4 + 4 x C/N) B per input sample"},
      "collective": rec["collective"], "nvlink": rec.get("nvlink"), "peer_store": rec.get("peer_store"),
      "e2e": {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
              "note": "host-buffer figure is reported by the stream-sharded run"},
    }
    print(json.dumps(line), flush=True)
  dist.barrier()
  dist.destroy_process_group()


def main():
  args = parse()
  if args.impl == "reference":
    run_reference(args)
  else:
    run_ours(args)


if __name__ == "__main__":
  main()
