#!/usr/bin/env python
"""bench.py — candidate variants/sec of the pileup-encode + CNN hot path on N B200s.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` (torchrun for
N>1, one rank per GPU); W untimed warm-up steps, then exactly K steps timed with CUDA events
between barriers; rank 0 prints ONE JSON line.

  step      one pass of the hot path over one batch of `--batch` synthetic candidate windows
            per GPU (config "HG002 chr20 30x WGS" stand-in: SURVEY.md §8(d) generator, 100x221x7).
  value     whole-job candidates/s, inputs resident in HBM.
  e2e       same metric through the host-buffer entry points (pinned host inputs, H2D + D2H
            inside the timed region).
  roofline  dominant kernel vs MEASURED_PEAKS.json; `roofline_encoder` is the HBM roofline of
            the pileup kernel (the "pileup HBM GB/s" half of the metric).
  cpu_baseline  the CPU oracle (faithful restatement of the reference algorithm) timed on a
            bounded sample on this box's host cores.

`--impl reference` times the reference-algorithm CPU path (oracle port; the reference itself
cannot be built here — DESIGN.md) on a bounded sample per step, rank 0 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

METRIC = 'candidate variants/sec (encode+CNN)'
UNIT = 'candidates/s'


def parse_args():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=8)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--batch', type=int, default=16384, help='candidate windows per step per GPU')
  ap.add_argument('--stage', default='auto', choices=['auto', 'encode', 'both'])
  ap.add_argument('--cpu-sample', type=int, default=2048, help='images in the bounded CPU sample')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-e2e', action='store_true')
  ap.add_argument('--no-extras', action='store_true', help='skip the parity / precision1 / config4 / config5 blocks')
  ap.add_argument('--parity-sample', type=int, default=48, help='windows of the last timed step re-derived on the CPU oracle')
  ap.add_argument('--config5-windows', type=int, default=10_000_000)
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write what the last timed step computed on rank 0 to DIR/<name>.npy as float32: probs.npy (every window, '
                       'a fixed sample when over 2^20) and images.npy (a fixed sample of 48 windows); the same arguments give the same inputs')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl == 'reference':
    ap.error('--dump-outputs writes the outputs of the CUDA path (--impl ours)')
  return args


def load_traffic():
  """Measured DRAM traffic per unit (ncu --set full captures; profiles/traffic.json) or {}."""
  p = os.path.join(ROOT, 'profiles', 'traffic.json')
  try:
    return json.load(open(p))
  except (OSError, ValueError):
    return {}


def load_peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    d = json.load(open(p))
    return {'hbm_gbs': d['hbm_gbs'], 'tflops': d['bf16_tflops'], 'tflops_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']),
            'source': 'measured (MEASURED_PEAKS.json)'}
  return {'hbm_gbs': 6650.0, 'tflops': 1590.0, 'tflops_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler:
  """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu_index):
    self.gpu = gpu_index
    self.lines = []
    self.proc = None

  def start(self):
    try:
      self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.gpu}', f'--query-gpu={self.Q}',
                                    '--format=csv,noheader,nounits', '-lms', '100'],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.t = threading.Thread(target=self._read, daemon=True)
      self.t.start()
    except OSError:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def stop(self):
    if not self.proc:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    time.sleep(0.15)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except subprocess.TimeoutExpired:
      self.proc.kill()
    sm, mx, reasons = [], [], set()
    for ln in self.lines:
      f = [x.strip() for x in ln.split(',')]
      if len(f) < 8:
        continue
      try:
        sm.append(float(f[1])); mx.append(float(f[2]))
      except ValueError:
        continue
      for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
        if v.lower().startswith('active'):
          reasons.add(name)
    sm.sort()
    return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(sm)}


def effective_cores():
  """Host cores this process may actually use: the scheduler affinity mask capped by the cgroup CPU quota
  (os.cpu_count() reports the machine, not the container)."""
  try:
    n = len(os.sched_getaffinity(0))
  except AttributeError:
    n = os.cpu_count() or 1
  try:
    quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
    if quota != 'max':
      n = min(n, max(1, int(float(quota) / float(period) + 0.999)))
  except (OSError, ValueError):
    try:   # cgroup v1
      quota = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
      period = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
      if quota > 0 and period > 0:
        n = min(n, max(1, (quota + period - 1) // period))
    except (OSError, ValueError):
      pass
  return max(1, n)


def wgs_options():
  from deepvariant_b200 import pileup_image as pi
  o = pi.default_options()
  o.channels = list(pi.PILEUP_CHANNELS_WITH_INSERT_SIZE)
  o.num_channels = 7
  return o


class CpuReference:
  """The reference algorithm on the host cores: C++ oracle port of the pileup encoder (one slice per
  thread; ctypes drops the GIL) followed by the torch fp32 Inception-v3 oracle (oneDNN, all cores)."""

  def __init__(self, params, cores):
    import torch
    import cnn_oracle
    import oracle_lib
    from deepvariant_b200 import modeling
    self.params, self.cores = params, cores
    oracle_lib.oracle()
    torch.set_num_threads(cores)
    self.cnn = cnn_oracle.FastCpuModel(modeling.random_weights(params.num_channels + params.num_alt_channels, 0))

  def encode(self, packed, n_images):
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    import oracle_lib
    from subbatch_util import take_images
    n_images = min(n_images, packed.n_images)
    threads = max(1, min(self.cores, n_images))
    parts = [take_images(packed, idx) for idx in np.array_split(np.arange(n_images), threads) if len(idx)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
      outs = list(ex.map(lambda pb: oracle_lib.encode_batch(self.params, pb), parts))
    return time.perf_counter() - t0, np.concatenate(outs)

  def classify(self, images, batch=128):
    import torch
    t0 = time.perf_counter()
    imgs = torch.from_numpy(images)
    for i in range(0, imgs.shape[0], batch):
      self.cnn.forward(imgs[i:i + batch])
    return time.perf_counter() - t0

  def tfexample_gzip_rate(self, images, n=96):
    """What the reference's make_examples pays on top of the pixels (SURVEY 8(d)): one tf.Example per image with the seven
    features of EncodeExample, written through the gzip TFRecord writer.  One core; returns examples/s per core."""
    import tempfile
    from deepvariant_b200 import protos, tfrecord
    n = min(n, len(images))
    variant = protos.Variant(reference_name='chr20', start=1000, end=1001, reference_bases='A', alternate_bases=['C']).serialize()
    idx = protos.encode_alt_allele_indices([0])
    with tempfile.TemporaryDirectory() as d:
      t0 = time.perf_counter()
      with tfrecord.Writer(os.path.join(d, 'ex.tfrecord.gz')) as w:
        for i in range(n):
          img = images[i]
          w.write(protos.encode_tf_example({
              'alt_allele_indices/encoded': ('bytes', [idx]), 'image/encoded': ('bytes', [img.tobytes()]),
              'image/shape': ('int64', list(img.shape)), 'locus': ('bytes', [b'chr20:1001-1001']), 'sequencing_type': ('int64', [0]),
              'variant/encoded': ('bytes', [variant]), 'variant_type': ('int64', [1])}))
      return n / (time.perf_counter() - t0)

  def calibrate(self, packed, target_s=4.0, lo=32, hi=4096):
    """Sample size so that one encode+classify pass takes about target_s seconds."""
    n0 = min(64, packed.n_images)
    te, imgs = self.encode(packed, n0)
    tc = self.classify(imgs)
    rate = n0 / max(te + tc, 1e-6)
    return int(max(lo, min(hi, packed.n_images, rate * target_s))), te, tc


def run_reference(args):
  """--impl reference: the reference algorithm's CPU path (oracle port), rank 0 only."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  from deepvariant_b200 import pileup_image as pi, synthetic
  params = pi.to_params(wgs_options())
  cores = effective_cores()
  ref = CpuReference(params, cores)
  packed = synthetic.make_batch(args.cpu_sample, 'cpu').to_packed()
  sample, _, _ = ref.calibrate(packed)
  times, te_sum, tc_sum = [], 0.0, 0.0
  for it in range(args.warmup + args.steps):
    te, imgs = ref.encode(packed, sample)
    tc = ref.classify(imgs)
    if it >= args.warmup:
      times.append(te + tc); te_sum += te; tc_sum += tc
  total = sum(times)
  value = sample * len(times) / total
  line = {
      'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': 1e3 * total / len(times), 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'u8 encode + f32 CNN', 'data': 'synthetic',
      'config': {'workload': 'HG002 chr20 30x WGS stand-in: synthetic 100x221x7 candidate windows (SURVEY 8d config 2/5)',
                 'stage': 'both', 'sample_images_per_step': sample},
      'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                       'sample': f'{sample} synthetic windows per step: C++ oracle port of pileup_image_native '
                                 f'({sample * len(times) / te_sum:.0f}/s) + torch fp32 CPU Inception-v3 '
                                 f'({sample * len(times) / tc_sum:.0f}/s); the reference itself is not buildable here'},
      'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }
  emit(line)


def ensure_built():
  """A fresh checkout has no built library (build artefacts are git-ignored): build in-tree with nvcc (rank 0 first)."""
  lib = os.path.join(ROOT, 'deepvariant_b200', 'csrc', 'libdvb.so')
  if os.path.exists(lib):
    return
  import __graft_entry__
  if int(os.environ.get('LOCAL_RANK', '0')) == 0:
    __graft_entry__.build()
  else:
    for _ in range(600):
      if os.path.exists(lib):
        time.sleep(2.0)
        return
      time.sleep(1.0)



def pacbio_options():
  """Config 4 (BASELINE.json: HG003 PacBio HiFi, --model_type=PACBIO): 100 x 147 x 10 (8 computed channels + 2 alt-aligned)."""
  from deepvariant_b200 import pileup_image as pi
  o = pi.default_options()
  o.channels = pi.PILEUP_DEFAULT_CHANNELS + ['haplotype', 'supplementary_alignment',
                                             'diff_channels_alternate_allele_1', 'diff_channels_alternate_allele_2']
  o.width = 147
  o.sort_by_haplotypes = True
  return o


def device_time_ms(stream, fn, steps, barrier):
  """CUDA-event time of `steps` calls of fn on `stream`, bracketed by barriers; returns ms per call."""
  import torch
  barrier()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record(stream)
  for _ in range(steps):
    fn()
  e1.record(stream)
  barrier()
  return e0.elapsed_time(e1) / steps


def max_over_ranks(x, dev, world):
  import torch
  import torch.distributed as dist
  t = torch.tensor([x], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  return float(t.item())


def parity_block(params, tb, images, probs, weights_seed, n_sample, probs_p1=None):
  """Untimed, after the timed loop: a spread of the LAST step's windows re-derived on the CPU oracle (tests/oracle_lib: C++
  restatement of pileup_image_native; tests/cnn_oracle: torch fp32 Inception-v3).  Images must be bit-exact."""
  import numpy as np
  import torch
  import cnn_oracle
  import oracle_lib
  from subbatch_util import take_images
  from deepvariant_b200 import modeling
  B = tb.n_images
  n_sample = max(3, min(n_sample, B))
  third = n_sample // 3
  idx = np.unique(np.r_[0:third, B // 2:B // 2 + third, B - (n_sample - 2 * third):B])
  packed = tb.to_packed()
  want_img = oracle_lib.encode_batch(params, take_images(packed, idx))
  got_img = images[torch.from_numpy(idx).to(images.device)].cpu().numpy()
  equal = int(sum(np.array_equal(got_img[i], want_img[i]) for i in range(len(idx))))
  out = {'images_checked': int(len(idx)), 'images_equal': equal, 'checker': 'oracle/dvb_oracle.cc (encoder, bit-exact) + tests/cnn_oracle.py (torch fp32)'}
  if probs is not None:
    w = modeling.random_weights(int(want_img.shape[3]), weights_seed)
    want_p = cnn_oracle.ReferenceModel(w).forward(torch.from_numpy(want_img)).numpy()
    got_p = probs[torch.from_numpy(idx).to(probs.device)].cpu().numpy()
    out.update({'precision': 0, 'max_abs_dp': float(np.abs(got_p - want_p).max()), 'tolerance_fp16_mode': 5e-3})
    if probs_p1 is not None:
      got1 = probs_p1[torch.from_numpy(idx).to(probs_p1.device)].cpu().numpy()
      out['max_abs_dp_precision1'] = float(np.abs(got1 - want_p).max())
      out['tolerance_precision1'] = 1e-5
  return out


DUMP_IMAGES = 48                 # 48 x 100 x 221 x 7 float32 = 30 MB
DUMP_MAX_PROB_ROWS = 1 << 20     # 12.6 MB of float32 probabilities


def _seeded_rows(n, k, seed=0):
  """All n rows when n <= k, else a fixed sorted sample of k of them."""
  import numpy as np
  if n <= k:
    return np.arange(n)
  return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_outputs(out_dir, images, probs):
  """Writes the last timed step's outputs, as a caller of the timed path receives them, to out_dir/<name>.npy in float32."""
  import numpy as np
  import torch
  os.makedirs(out_dir, exist_ok=True)
  arrays = {'images': (images, DUMP_IMAGES)}
  if probs is not None:
    arrays['probs'] = (probs, DUMP_MAX_PROB_ROWS)
  shapes = {}
  for name, (t, k) in arrays.items():
    rows = torch.from_numpy(_seeded_rows(t.shape[0], k)).to(t.device)
    a = t.index_select(0, rows).cpu().numpy().astype(np.float32)
    np.save(os.path.join(out_dir, name + '.npy'), a)
    shapes[name] = list(a.shape)
  return shapes


_REAL_STDOUT = None


def emit(line: dict) -> None:
  """The ONE JSON line of the contract, on the process's real stdout."""
  out = _REAL_STDOUT or sys.stdout
  print(json.dumps(line), file=out, flush=True)


def main():
  global _REAL_STDOUT
  args = parse_args()
  # Libraries write banners to stdout (NCCL prints its version line there): keep the real stdout for the JSON line only
  # and send everything else to stderr.
  sys.stdout.flush()
  _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
  os.dup2(2, 1)
  ensure_built()
  if args.impl == 'reference':
    run_reference(args)
    return
  import torch
  import torch.distributed as dist
  import numpy as np
  from deepvariant_b200 import call_variants as cv, pileup_image as pi, synthetic

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)
  peaks = load_peaks()

  o = wgs_options()
  params = pi.to_params(o)
  enc = pi.GpuEncoder(params, device=local)
  B = args.batch
  # Region sharding: every rank owns its own candidate windows (chunk = rank); no exchange.
  tb = synthetic.make_batch(B, dev, chunk=rank)
  images = torch.empty((B,) + enc.shape, dtype=torch.uint8, device=dev)

  cnn = None
  stage = args.stage
  if stage in ('auto', 'both'):
    try:
      cnn = cv.GpuCnn.random_init(enc.shape, device=local, max_batch=B)
      stage = 'both'
    except (ImportError, AttributeError) as e:
      if stage == 'both':
        raise
      stage = 'encode'
  probs = torch.empty((B, 3), dtype=torch.float32, device=dev) if cnn else None
  stream = torch.cuda.current_stream()

  def step():
    enc.encode_device(tb, images, stream=stream)
    if cnn:
      cnn.forward_device(images, probs, stream=stream)

  def barrier():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  for _ in range(args.warmup):
    step()
  enc.check()
  barrier()
  l0 = enc.launch_count + (cnn.launch_count if cnn else 0)
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  # per-kernel-group device time of the encoder, on the launching stream
  enc_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
  e0.record(stream)
  for k in range(args.steps):
    enc_ev[k][0].record(stream)
    enc.encode_device(tb, images, stream=stream)
    enc_ev[k][1].record(stream)
    if cnn:
      cnn.forward_device(images, probs, stream=stream)
  e1.record(stream)
  barrier()
  clocks = sampler.stop() if rank == 0 else None
  enc.check()
  # Later blocks reuse `images` and `probs`: save the timed step's outputs before they run.
  dumped = dump_outputs(args.dump_outputs, images, probs) if args.dump_outputs and rank == 0 else None
  ms_total = e0.elapsed_time(e1)
  launches = enc.launch_count + (cnn.launch_count if cnn else 0) - l0
  enc_ms = sum(a.elapsed_time(b) for a, b in enc_ev) / args.steps
  t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_total = float(t.item())
  ms_step = ms_total / args.steps
  value = world * B / (ms_step * 1e-3)

  # ---- e2e: pinned host inputs -> H2D -> hot path -> D2H, through the same entry points ----
  e2e = None
  if not args.no_e2e:
    host = tb.to('cpu').pin()       # the caller's batch, in pinned host memory
    h2d = host.input_bytes()
    if cnn:
      out_host = torch.empty((B, 3), dtype=torch.float32).pin_memory()
      out_np = out_host.numpy()
      d2h = out_host.numel() * 4 + B * 4     # probabilities + rows_kept
    else:
      out_host = torch.empty((B,) + enc.shape, dtype=torch.uint8).pin_memory()
      d2h = out_host.numel()

    def e2e_step():
      # The reference-facing call: HOST DvbBatch in, host result out, through the C ABI
      # (dvb_encode_classify_host: validate + H2D + encode + CNN + D2H + synchronise).
      if cnn:
        enc.encode_classify_host(host, cnn, out_np)
        return None
      d = host.to(dev, non_blocking=True)
      enc.encode_device(d, images, stream=stream)
      out_host.copy_(images, non_blocking=True)
      return d

    keep = [e2e_step() for _ in range(max(1, args.warmup // 2))]
    barrier()
    n_e2e = max(2, args.steps // 2)
    # The host entry point runs on the handle's own stream and synchronises before it returns, so the
    # timed region is bracketed by host clocks around fully synchronous calls (plus device syncs).
    t_a = time.perf_counter()
    for _ in range(n_e2e):
      keep.append(e2e_step())
    torch.cuda.synchronize()
    t_b = time.perf_counter()
    barrier()
    t2 = torch.tensor([(t_b - t_a) * 1e3 / n_e2e], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e = {'value': world * B / (float(t2.item()) * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
           'd2h_bytes_per_step': d2h, 'steps': n_e2e,
           'api': 'dvb_encode_classify_host (C ABI, pinned host DvbBatch in, host probabilities out, synchronous)' if cnn else 'device entry points + torch copies'}
    del keep

  # ---- extras (all ranks take part in the timed parts; rank 0 reports): precision 1, config 4, config 5, parity ----
  extras = {}
  if not args.no_extras:
    k_x = max(2, args.steps // 4)
    if cnn:
      # (1) precision 1 = split-fp16 x3, the mode that meets the north star's 1e-5: same step, same windows
      cnn1 = cv.GpuCnn.random_init(enc.shape, device=local, max_batch=min(B, 2048), precision=1)
      probs1 = torch.empty((B, 3), dtype=torch.float32, device=dev)

      def step1():
        enc.encode_device(tb, images, stream=stream)
        cnn1.forward_device(images, probs1, stream=stream)
      step1()
      ms1 = max_over_ranks(device_time_ms(stream, step1, k_x, barrier), dev, world)
      p1 = {'value': world * B / (ms1 * 1e-3), 'unit': UNIT, 'ms_per_step': ms1, 'steps': k_x,
            'dtype': 'u8 encode + split-fp16 x3 CNN (fp32-grade products, fp32 accumulate)'}
      if e2e is not None:
        out1 = np.empty((B, 3), dtype=np.float32)
        enc.encode_classify_host(host, cnn1, out1)
        barrier()
        t_a = time.perf_counter()
        for _ in range(k_x):
          enc.encode_classify_host(host, cnn1, out1)
        torch.cuda.synchronize()
        t_e = max_over_ranks((time.perf_counter() - t_a) * 1e3 / k_x, dev, world)
        barrier()
        p1['e2e'] = {'value': world * B / (t_e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'steps': k_x}
      extras['precision1'] = p1
    # (2) config 5: encode-only sweep over --config5-windows candidate windows (several distinct chunks, cycled)
    n_launch = max(1, (args.config5_windows + B - 1) // B)
    chunks = [tb] + [synthetic.make_batch(B, dev, chunk=world * (1 + j) + rank) for j in range(2)]
    it = [0]

    def enc_only():
      enc.encode_device(chunks[it[0] % len(chunks)], images, stream=stream)
      it[0] += 1
    enc_only()
    ms5 = max_over_ranks(device_time_ms(stream, enc_only, n_launch, barrier), dev, world)
    enc.check()
    ab5 = sum(c.algorithmic_bytes(enc.image_bytes, o.width) for c in chunks) / len(chunks)
    extras['config5_encode_only'] = {
        'n_windows': world * n_launch * B, 'windows_per_s': world * B / (ms5 * 1e-3), 'ms_per_launch': ms5, 'launches_per_gpu': n_launch,
        'gbs_per_gpu': ab5 / (ms5 * 1e-3) / 1e9, 'frac': ab5 / (ms5 * 1e-3) / 1e9 / peaks['hbm_gbs'], 'peak': peaks['hbm_gbs'],
        'workload': 'synthetic 30x reads, 100x221x7 windows, %d distinct chunks of %d cycled' % (len(chunks), B)}
    del chunks
    # (3) config 4: PACBIO layout (100 x 147 x 10), encode + classify on long-read-shaped synthetic windows
    if cnn:
      o4 = pacbio_options()
      params4 = pi.to_params(o4)
      enc4 = pi.GpuEncoder(params4, device=local)
      tb4 = synthetic.make_batch(B, dev, chunk=rank, width=o4.width, hp=True)
      images4 = torch.empty((B,) + enc4.shape, dtype=torch.uint8, device=dev)
      cnn4 = cv.GpuCnn.random_init(enc4.shape, device=local, max_batch=B)
      probs4 = torch.empty((B, 3), dtype=torch.float32, device=dev)

      def enc4_only():
        enc4.encode_device(tb4, images4, stream=stream)

      def step4():
        enc4.encode_device(tb4, images4, stream=stream)
        cnn4.forward_device(images4, probs4, stream=stream)
      step4()
      ms4 = max_over_ranks(device_time_ms(stream, step4, k_x, barrier), dev, world)
      ms4e = max_over_ranks(device_time_ms(stream, enc4_only, 4 * k_x, barrier), dev, world)
      enc4.check()
      ab4 = tb4.algorithmic_bytes(enc4.image_bytes, o4.width)
      r4 = cnn4.roofline(ms4 - ms4e, B, peaks)
      extras['config4_pacbio'] = {
          'value': world * B / (ms4 * 1e-3), 'unit': UNIT, 'ms_per_step': ms4, 'steps': k_x, 'image_shape': list(enc4.shape),
          'roofline': {k: r4[k] for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'flops_per_image', 'ms_cnn_per_step')},
          'roofline_encoder': {'bound': 'hbm', 'achieved': ab4 / (ms4e * 1e-3) / 1e9, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                               'frac': ab4 / (ms4e * 1e-3) / 1e9 / peaks['hbm_gbs'], 'ms_per_launch': ms4e,
                               'windows_per_s_encode_only': B / (ms4e * 1e-3)}}
      if rank == 0:
        extras['config4_pacbio']['parity'] = parity_block(params4, tb4, images4, probs4, 0, min(args.parity_sample, 24))
      cnn4.close(); enc4.close()
      del images4, tb4
    # (4) parity of what was just timed: the last step's images / probabilities against the CPU oracle
    if rank == 0:
      step()
      if cnn:
        cnn1.forward_device(images, probs1, stream=stream)
      torch.cuda.synchronize()
      extras['parity'] = parity_block(params, tb, images, probs, 0, args.parity_sample, probs1 if cnn else None)
      if cnn and 'precision1' in extras:
        extras['precision1']['max_abs_dp'] = extras['parity'].get('max_abs_dp_precision1')
    if cnn:
      cnn1.close()
    barrier()

  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return

  # ---- rooflines ----
  alg_bytes = tb.algorithmic_bytes(enc.image_bytes, o.width)
  enc_gbs = alg_bytes / (enc_ms * 1e-3) / 1e9
  traffic = load_traffic()
  enc_traffic = traffic.get('encoder', {}).get('dram_bytes_per_window')
  roof_enc = {'bound': 'hbm', 'kernel': 'dvb_encode_kernel', 'achieved': enc_gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
              'frac': enc_gbs / peaks['hbm_gbs'], 'traffic': enc_traffic * B if enc_traffic else None,
              'traffic_source': traffic.get('encoder', {}).get('capture'), 'peak_source': peaks['source'],
              'ms_per_launch': enc_ms, 'algorithmic_bytes_per_launch': alg_bytes,
              'windows_per_s_encode_only': B / (enc_ms * 1e-3)}
  # The kernel writes 36 bytes for every byte it reads, and HBM3e takes a pure write stream at about 60 % of its copy rate: the
  # write-only ceiling is measured here, on this GPU, with cudaMemset over the image buffer (reported beside `peak`, not instead of it).
  try:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flat = images.view(-1)
    for _ in range(2):
      flat.zero_()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
      flat.zero_()
    e1.record()
    torch.cuda.synchronize()
    wc = 5 * flat.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9
    roof_enc['write_only_ceiling'] = {'gbs': wc, 'frac_of_it': enc_gbs / wc, 'how': f'cudaMemset of the {flat.numel() >> 20} MiB image buffer, 5 runs, CUDA events'}
  except Exception as e:   # pylint: disable=broad-except
    roof_enc['write_only_ceiling'] = {'error': str(e)[:120]}
  if cnn:
    roofline = cnn.roofline(ms_step - enc_ms, B, peaks)
    cnn_traffic = traffic.get('cnn', {}).get('dram_bytes_per_image')
    roofline['traffic'] = cnn_traffic * B if cnn_traffic else None
    roofline['traffic_source'] = traffic.get('cnn', {}).get('capture')
  else:
    roofline = roof_enc

  cpu_baseline = None
  if not args.no_cpu_baseline:
    cores = effective_cores()
    ref = CpuReference(params, cores)
    packed = synthetic.make_batch(args.cpu_sample, 'cpu').to_packed()
    sample, _, _ = ref.calibrate(packed, target_s=6.0)
    te, imgs = ref.encode(packed, sample)
    reps = 1
    while te < 1.0 and reps < 64:   # the encoder sample is cheap: repeat it to get a stable rate
      t2, _ = ref.encode(packed, sample)
      te += t2; reps += 1
    tc = ref.classify(imgs)
    r_enc, r_cnn = sample * reps / te, sample / tc
    r_gz = ref.tfexample_gzip_rate(imgs)
    cpu_baseline = {'value': 1.0 / (1.0 / r_enc + 1.0 / r_cnn), 'unit': UNIT, 'cores': cores, 'kind': 'port',
                    'tfexample_gzip_examples_per_s_per_core': r_gz,
                    'sample': f'{sample} synthetic windows: C++ oracle port of pileup_image_native.cc {r_enc:.0f}/s '
                              f'({te:.1f} s) then torch fp32 CPU Inception-v3 {r_cnn:.0f}/s ({tc:.1f} s) on the same cores',
                    'encode_only': r_enc, 'cnn_only': r_cnn}

  line = {
      'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'u8' if not cnn else 'u8 encode + fp16 CNN (fp32 accumulate)', 'data': 'synthetic',
      'config': {'workload': 'HG002 chr20 30x WGS stand-in: synthetic 100x221x7 candidate windows (SURVEY 8d config 2/5)',
                 'stage': stage, 'batch_per_gpu': B, 'image_shape': list(enc.shape),
                 'l2': 'working set per step (inputs %.0f MB, images %.0f MB) exceeds the 126 MB L2' %
                       (tb.input_bytes() / 1e6, B * enc.image_bytes / 1e6),
                 'sharding': 'candidates region-sharded across ranks, no collective'},
      'gpu_launches': launches, 'clocks': clocks, 'e2e': e2e, 'roofline': roofline, 'roofline_encoder': roof_enc,
      'cpu_baseline': cpu_baseline,
  }
  if dumped:
    line['dump_outputs'] = {'dir': args.dump_outputs, 'arrays': dumped}
  line.update(extras)
  emit(line)
  if world > 1:
    dist.destroy_process_group()


if __name__ == '__main__':
  main()
