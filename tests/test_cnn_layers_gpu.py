"""Every classifier layer against a float64 restatement of that layer, computed from the layer's own operands.

The end-to-end tests (test_cnn_gpu.py) compare block outputs with the fp32 oracle at max|error| / max|tensor| < 2e-2: fp16
rounding compounds over 94 layers, so that bar has to be loose, and a fault in one layer fades into it.  Here each layer is
checked in isolation.  Its input is the engine's own fp16 activation (dvb_cnn_debug_tensor), its weights are the fp16 values
of the weights blob, its bias the blob's fp32 bias, so the only difference a correct kernel may show is fp32 accumulation
error plus one rounding of the output.  Per element:

  precision 0   |got - ref| <= 2^-11 |ref| + (K + 1) 2^-23 S + 2^-24

      ref = relu(conv(x, W) + b) in float64, S = conv(|x|, |W|) + |b|, K = kh kw cin.  The products of two fp16 numbers are
      exact in fp32, so the K products and the bias are summed with (K + 1)-term fp32 error: at most (K + 1) u S.  Tensor
      cores align and truncate (round toward zero) where IEEE addition rounds to nearest (Fasi et al., "Numerical behavior of
      NVIDIA tensor cores", 2021), so u = 2^-23 rather than 2^-24.  The ReLU is exact; rounding to fp16 adds at most 2^-11 of
      the value (2^-11 |ref| plus 2^-11 of the accumulation error, which the 2^-24 term and the slack of (K + 1) cover) and,
      below 2^-14, half the subnormal spacing, 2^-25.

  precision 1   |got - ref| <= 2^-21 |ref| + (K + 4) 2^-23 S + 2^-30,  i.e. c 2^-21 S + 2^-21 |ref| with c = (K + 4) / 4

      Operands are split pairs, A = Am + Ar 2^-11 with |Ar 2^-11| <= 2^-11 |A| (the blob's residual plane for the weights,
      the tensor's residual plane for the activations).  The kernel sums Am Bm + (Am Br + Ar Bm) 2^-11 and drops
      Ar Br 2^-22: at most 2^-22 S = 2 2^-23 S.  The main products accumulate with K 2^-23 S as above; the cross terms
      are 2^-11 smaller and add 2K 2^-23 2S 2^-11 < 2^-23 S; combining the two accumulators and adding the bias round twice
      in fp32 (2^-23 S).  The activation this test reads, fp32(main + res 2^-11), is itself within 2^-24 of the pair the
      kernel multiplied (2^-24 S more).  Total (K + 4) 2^-23 S.  The output is stored as a pair again: main = fp16(v),
      res = fp16((v - main) 2^11) keeps v to 2^-22, and reading it back as fp32 adds 2^-24: below 2^-21 |v|.

  pools         3x3 average: <= 12 fp32 roundings over S = avgpool(|x|) (+ |b| when the pool carries its convolution's
                bias), then the output rounding as above.  Max pools at precision 0: bit-equal to the max of the fp16 input;
                at precision 1 the split store keeps the maximum to 2^-21.
  tail          pooled = mean of the fp16 mixed10 to (hw + 4) 2^-24 mean|x|; probabilities = float64 softmax of the
                engine's own pooled features, within 1e-6.

Besides the bound, each precision-0 convolution and average pool must match fp16(ref) (the correctly rounded value) in at
least CR_FLOOR of its elements: an accumulation off by more than the usual last fp32 bits, or a rounding mode other than
round-to-nearest, shows up there first.

The checker walks modeling.inception_v3_graph in the engine's order (the 1x1 convolution behind each average pool runs
first under DVB_CNN_POOL_AFTER_CONV=1, the default; conv3's epilogue applies the max pool behind it under DVB_CNN_FUSE_POOL=1,
so 's3' is checked through 'p1') and counts what it verified: 94 convolutions, 4 max pools, 9 average pools, pooled
features and probabilities.  A tensor the engine should have but does not return is an error, not a skip.

The CPU tests at the end run the checker on Fp16Engine, a torch emulation of an fp16 engine (fp16 operands, fp32
accumulation, round-to-nearest output per layer), and on mutated copies of it.  Measured on that emulation (100x221x7,
modeling.random_weights(7, 1), two random images), the old end-to-end bar (stem 6e-3, blocks and branch tensors 2e-2 of
scale, probabilities 5e-3 from the fp32 oracle) against the layer checker:

  mutant                                                        old bar                            layer checker
  conv42 (mixed5_s1, merged 1x1 member): one bias dropped       passes (worst 2.2e-3, p 6.9e-5)    fails at conv42 (29x the bound)
  conv49 (mixed5[384:576]): one bias dropped                    passes (worst 1.1e-2, p 3.4e-4)    fails at conv49 (44x)
  conv17 (mixed1_d2, 3x3 same): tap (0, 0) dropped, last row    fails  (worst 0.21,   p 2.9e-3)    fails at conv17 (1.8e3x)
  conv34 (mixed4[192:384], 7x1): last image from the previous   fails  (worst 0.20,   p 5.4e-3)    fails at conv34 (470x)
  every output truncated to fp16 instead of rounded             passes (worst 9.0e-3, p 3.0e-3)    fails at conv1 (1.9x)
  conv42 written one channel off                                fails  (worst 0.78,   p 2.2e-2)    fails at conv42 (3.1e3x)

(worst = largest block or branch error of scale, p = largest probability error.)  The two one-channel bias faults and the
truncating conversion pass every threshold of the end-to-end tests.

OLD_BAR_VERDICT below holds the same table; test_old_end_to_end_bar_misses_what_the_layer_checker_catches keeps it true.
"""
from __future__ import annotations

import dataclasses
import re
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from deepvariant_b200 import modeling

CR_FLOOR = 0.97        # correctly rounded fraction per precision-0 layer (measured: see the report printed with -s, DESIGN.md 5)
PROBS_TOL = 1e-6
GEOMETRIES = [(100, 221, 7), (100, 147, 10), (100, 221, 6), (100, 221, 9), (140, 221, 7)]


# ---- the engine's operands ----------------------------------------------------------------------------------------------------

@dataclasses.dataclass
class BlobParams:
  convs: List[tuple]        # (W float64 [cout][cin][kh][kw], b float64 [cout]) per convolution, network order
  dense_kernel: torch.Tensor
  dense_bias: torch.Tensor
  precision: int


def parse_blob(blob: bytes) -> BlobParams:
  """The weights exactly as dvb_cnn_create receives them: fp16 kernels (+ residual plane 2^-11 at precision 1), fp32 bias."""
  magic, _, n_conv = np.frombuffer(blob, '<i4', 3, 0)
  split = int(magic) == modeling.BLOB_MAGIC_SPLIT
  pos = 12
  convs = []
  for _ in range(int(n_conv)):
    kh, kw, cin, cp, cout = (int(v) for v in np.frombuffer(blob, '<i4', 5, pos))
    pos += 20
    cnt = cout * kh * kw * cp
    w = np.frombuffer(blob, '<f2', cnt, pos).reshape(cout, kh, kw, cp)[..., :cin].astype(np.float64)
    pos += 2 * cnt
    if split:
      w = w + np.frombuffer(blob, '<f2', cnt, pos).reshape(cout, kh, kw, cp)[..., :cin].astype(np.float64) / modeling.SPLIT_SCALE
      pos += 2 * cnt
    b = np.frombuffer(blob, '<f4', cout, pos).astype(np.float64)
    pos += 4 * cout
    convs.append((torch.from_numpy(np.ascontiguousarray(w.transpose(0, 3, 1, 2))), torch.from_numpy(b)))
  dk = np.frombuffer(blob, '<f4', 2048 * 3, pos).reshape(2048, 3).astype(np.float64)
  pos += 4 * 2048 * 3
  db = np.frombuffer(blob, '<f4', 3, pos).astype(np.float64)
  assert pos + 12 == len(blob)
  return BlobParams(convs, torch.from_numpy(dk), torch.from_numpy(db), 1 if split else 0)


@dataclasses.dataclass
class Route:
  precision: int = 0
  pool_after_conv: bool = True   # DVB_CNN_POOL_AFTER_CONV: the 1x1 convolution behind an average pool runs first
  fused_pool: bool = True        # conv3 + max pool in conv_rows_kernel's epilogue: 's3' is not materialised


@dataclasses.dataclass
class Step:
  kind: str                      # 'conv' | 'conv+maxpool' | 'maxpool' | 'avgpool'
  op: modeling.Op
  ci: int = -1                   # convolution index (blob order); for a pool that carries a bias: the conv it came from
  pool: Optional[modeling.Op] = None
  no_act: bool = False           # raw accumulator out (the pool behind it adds the bias and the ReLU)


def engine_steps(C: int, route: Route) -> List[Step]:
  """modeling.inception_v3_graph in the order and form the engine runs it."""
  ops, _ = modeling.inception_v3_graph(C)
  steps: List[Step] = []
  ci = 0
  i = 0
  while i < len(ops):
    o = ops[i]
    nx = ops[i + 1] if i + 1 < len(ops) else None
    if (route.pool_after_conv and o.kind == 'avgpool' and nx is not None and nx.kind == 'conv' and nx.kh == 1 and nx.kw == 1 and
        nx.stride == 1 and nx.src == o.dst):
      steps.append(Step('conv', dataclasses.replace(nx, src=o.src, dst=o.dst, dst_channel_offset=0), ci, no_act=True))
      steps.append(Step('avgpool', dataclasses.replace(o, src=o.dst, dst=nx.dst, dst_channel_offset=nx.dst_channel_offset,
                                                       cin=nx.cout, cout=nx.cout), ci))
      ci += 1
      i += 2
    elif route.fused_pool and o.kind == 'conv' and o.dst == 's3':
      assert nx.kind == 'maxpool' and nx.src == 's3'
      steps.append(Step('conv+maxpool', o, ci, pool=nx))
      ci += 1
      i += 2
    elif o.kind == 'conv':
      steps.append(Step('conv', o, ci))
      ci += 1
      i += 1
    else:
      steps.append(Step(o.kind, o))
      i += 1
  assert ci == 94
  return steps


# ---- the checker ---------------------------------------------------------------------------------------------------------------

def _conv(x, w, op):
  pad = ((op.kh - 1) // 2, (op.kw - 1) // 2) if op.same else (0, 0)
  return F.conv2d(x, w, None, stride=op.stride, padding=pad)


def _avgpool(x):
  return F.avg_pool2d(x, 3, 1, 1, count_include_pad=False)   # TF 'same': padding excluded from the divisor


class LayerChecker:
  """Walks the graph after one forward and checks every op against float64 from the engine's own operands.

  get(name) -> float32 [n, H, W, C] of the first n images (the engine's debug copy; 'pooled' -> [n, 1, 1, 2048]);
  idx = the images to check (the float64 work is done for those only); from_tensor: start at the first op reading it."""

  def __init__(self, get: Callable[[str], np.ndarray], blob: bytes, images: np.ndarray, probs: np.ndarray, idx: Sequence[int],
               route: Route, from_tensor: Optional[str] = None):
    self.get, self.images, self.probs, self.idx, self.route = get, images, probs, list(idx), route
    self.C = images.shape[3]
    self.params = parse_blob(blob)
    assert self.params.precision == route.precision
    self.from_tensor = from_tensor
    self.cache: Dict[str, torch.Tensor] = {}
    self.report: List[tuple] = []         # (label, worst |got - ref| / bound, correctly rounded fraction or None)
    self.failures: List[str] = []
    self.counts = {'conv': 0, 'maxpool': 0, 'avgpool': 0, 'pooled': 0, 'probs': 0}

  # float64 NCHW of the checked images
  def t(self, name: str) -> torch.Tensor:
    if name not in self.cache:
      a = self.get(name)
      self.cache[name] = torch.from_numpy(np.ascontiguousarray(a[self.idx])).to(torch.float64).permute(0, 3, 1, 2)
    return self.cache[name]

  def out_bound(self, ref):
    return (2.0 ** -11 if self.route.precision == 0 else 2.0 ** -21) * ref.abs() + (2.0 ** -24 if self.route.precision == 0 else 2.0 ** -30)

  def conv_bound(self, ref, S, K):
    k = K + 1 if self.route.precision == 0 else K + 4
    return self.out_bound(ref) + k * 2.0 ** -23 * S

  def pool_bound(self, ref, S):
    return self.out_bound(ref) + 12 * 2.0 ** -24 * S

  def compare(self, label, got, ref, bound, rounded=True):
    assert got.shape == ref.shape, (label, tuple(got.shape), tuple(ref.shape))
    err = (got - ref).abs()
    worst = float((err / bound).max())
    cr = None
    if self.route.precision == 0 and rounded:
      cr = float((got.numpy() == ref.numpy().astype(np.float16).astype(np.float64)).mean())
    self.report.append((label, worst, cr))
    if not worst <= 1.0:
      at = np.unravel_index(int((err / bound).argmax()), tuple(err.shape))
      self.failures.append(f'{label}: |got - ref| / bound = {worst:.3g} at [image {self.idx[at[0]]}, c {at[1]}, h {at[2]}, w {at[3]}]')
    elif cr is not None and cr < CR_FLOOR:
      self.failures.append(f'{label}: only {cr:.4f} of the elements are fp16(ref)')

  def conv_ref(self, step: Step, x):
    w, b = self.params.convs[step.ci]
    op = step.op
    acc, S = _conv(x, w, op), _conv(x.abs(), w.abs(), op)
    if step.no_act:
      return acc, S
    return torch.relu(acc + b.view(1, -1, 1, 1)), S + b.abs().view(1, -1, 1, 1)

  def dst(self, op, c):
    return self.t(op.dst)[:, op.dst_channel_offset:op.dst_channel_offset + c]

  def run(self):
    steps = engine_steps(self.C, self.route)
    if self.from_tensor is not None:
      steps = steps[next(i for i, s in enumerate(steps) if s.op.src == self.from_tensor):]
    for s in steps:
      op = s.op
      label = f'conv{s.ci + 1} -> {op.dst}[{op.dst_channel_offset}:{op.dst_channel_offset + op.cout}]' if 'conv' in s.kind else \
              f'{s.kind} {op.src} -> {op.dst}[{op.dst_channel_offset}:{op.dst_channel_offset + op.cout}]'
      if s.kind in ('conv', 'conv+maxpool'):
        if s.ci == 0:
          x = torch.from_numpy(self.images[self.idx]).to(torch.float64).permute(0, 3, 1, 2)
          x = (x - 128.0) / 128.0      # exact in fp16
        else:
          x = self.t(op.src)
        ref, S = self.conv_ref(s, x)
        bound = self.conv_bound(ref, S, op.kh * op.kw * op.cin)
        if s.kind == 'conv':
          self.compare(label + (' (no bias, no ReLU)' if s.no_act else ''), self.dst(op, op.cout), ref, bound)
        else:
          # rounding is monotone, so it commutes with the max: fp16(max ref) = max fp16(ref), and the error of a max is at most
          # the largest error under the window
          try:
            self.get('s3')
            self.failures.append('s3 is materialised: conv3 + max pool did not run fused')
          except Exception:  # pylint: disable=broad-except
            pass
          p = s.pool
          self.compare(label + f' + maxpool -> {p.dst}', self.dst(p, op.cout), F.max_pool2d(ref, 3, 2), F.max_pool2d(bound, 3, 2))
          self.counts['maxpool'] += 1
        self.counts['conv'] += 1
      elif s.kind == 'maxpool':
        x = self.t(op.src)
        ref = F.max_pool2d(x, 3, 2)
        got = self.dst(op, op.cout)
        if self.route.precision == 0:
          same = bool(torch.equal(got, ref))
          self.report.append((label, 0.0 if same else float('inf'), 1.0 if same else float((got == ref).double().mean())))
          if not same:
            self.failures.append(f'{label}: not bit-equal to the max of its fp16 input')
        else:
          self.compare(label, got, ref, self.out_bound(ref), rounded=False)
        self.counts['maxpool'] += 1
      else:
        x = self.t(op.src)
        ref, S = _avgpool(x), _avgpool(x.abs())
        if s.ci >= 0:          # behind its 1x1 convolution: + bias, ReLU
          b = self.params.convs[s.ci][1].view(1, -1, 1, 1)
          ref, S = torch.relu(ref + b), S + b.abs()
        self.compare(label + (' + bias, ReLU' if s.ci >= 0 else ''), self.dst(op, op.cout), ref, self.pool_bound(ref, S))
        self.counts['avgpool'] += 1
    self.check_tail()
    return self

  def check_tail(self):
    feat = self.t('mixed10')
    hw = feat.shape[2] * feat.shape[3]
    ref = feat.mean(dim=(2, 3))
    bound = (hw + 4) * 2.0 ** -24 * feat.abs().mean(dim=(2, 3)) + 2.0 ** -60
    got = torch.from_numpy(self.get('pooled')[self.idx].reshape(len(self.idx), -1)).to(torch.float64)
    worst = float(((got - ref).abs() / bound).max())
    self.report.append(('pooled = mean(mixed10)', worst, None))
    if not worst <= 1.0:
      self.failures.append(f'pooled: |got - ref| / bound = {worst:.3g}')
    self.counts['pooled'] += 1
    want = torch.softmax(got @ self.params.dense_kernel + self.params.dense_bias, dim=1)
    err = float((torch.from_numpy(self.probs[self.idx]).to(torch.float64) - want).abs().max())
    self.report.append(('probs = softmax(pooled . dense)', err / PROBS_TOL, None))
    if not err <= PROBS_TOL:
      self.failures.append(f'probs: |got - float64 softmax| = {err:.3g}')
    self.counts['probs'] += 1

  def expected_counts(self):
    """Every op of the graph from the first one checked: convolutions, max and average pools (whatever form the route ran
    them in), pooled features and probabilities."""
    ops, _ = modeling.inception_v3_graph(self.C)
    first = ops.index(next(o for o in ops if o.src == self.from_tensor)) if self.from_tensor else 0
    rest = ops[first:]
    return {'conv': sum(o.kind == 'conv' for o in rest), 'maxpool': sum(o.kind == 'maxpool' for o in rest),
            'avgpool': sum(o.kind == 'avgpool' for o in rest), 'pooled': 1, 'probs': 1}

  def print_report(self, title):
    print(f'\n== {title}: {len(self.report)} checks on images {self.idx}')
    for label, worst, cr in self.report:
      print(f'  {label:58s} worst/bound {worst:8.3g}' + (f'   fp16(ref) {cr:.5f}' if cr is not None else ''))

  def assert_ok(self, title=''):
    self.print_report(title)
    assert not self.failures, '\n'.join(self.failures)
    want = self.expected_counts()
    assert self.counts == want, (self.counts, want)


# ---- an fp16 engine on the CPU (checks the checker) ------------------------------------------------------------------------------

@dataclasses.dataclass
class Mutant:
  name: str
  conv: Optional[str] = None     # modeling op name ('conv42') the fault sits in
  fault: str = ''                # 'drop_bias' | 'drop_tap' | 'prev_image' | 'truncate' | 'channel_off'


def _truncate_to_fp16(y: torch.Tensor) -> torch.Tensor:
  h = y.half()
  over = h.float().abs() > y.abs()
  bits = h.view(torch.int16).clone()
  bits[over] -= 1               # sign-magnitude: one unit less magnitude = one ulp toward zero
  return bits.view(torch.float16).float()


class Fp16Engine:
  """fp16 activations and weights, fp32 accumulation (torch's CPU convolution), round-to-nearest to fp16 per stored tensor;
  materialises what the CUDA engine's default plan materialises (debug_tensor)."""

  def __init__(self, blob: bytes, C: int, mutant: Optional[Mutant] = None):
    p = parse_blob(blob)
    self.convs = [(w.float(), b.float()) for w, b in p.convs]
    self.dk, self.db = p.dense_kernel.float(), p.dense_bias.float()
    self.C = C
    self.mutant = mutant or Mutant('none')
    self.tensors: Dict[str, torch.Tensor] = {}

  def _round(self, y):
    return _truncate_to_fp16(y) if self.mutant.fault == 'truncate' else y.half().float()

  def forward_host(self, images: np.ndarray) -> np.ndarray:
    _, ch = modeling.inception_v3_graph(self.C)
    m = self.mutant
    t: Dict[str, torch.Tensor] = {}
    n = images.shape[0]

    def store(name, off, y, total):
      if name not in t:
        t[name] = torch.zeros((n, total) + tuple(y.shape[2:]))
      t[name][:, off:off + y.shape[1]] = y

    x0 = ((torch.from_numpy(images).float() - 128.0) / 128.0).permute(0, 3, 1, 2)
    for s in engine_steps(self.C, Route()):
      op = s.op
      if 'conv' in s.kind:
        w, b = self.convs[s.ci]
        x = x0 if s.ci == 0 else t[op.src]
        if m.conv == op.name and m.fault == 'prev_image':
          x = x.clone()
          x[-1] = x[-2]
        if m.conv == op.name and m.fault == 'drop_bias':
          b = b.clone()
          b[int(np.argsort(np.abs(b.numpy()))[len(b) // 2])] = 0.0     # the channel of median |bias|
        y = _conv(x, w, op)
        if m.conv == op.name and m.fault == 'drop_tap':
          wt = torch.zeros_like(w)
          wt[:, :, 0, 0] = w[:, :, 0, 0]
          y[:, :, -1, :] -= _conv(x, wt, op)[:, :, -1, :]
        if not s.no_act:
          y = torch.relu(y + b.view(1, -1, 1, 1))
        y = self._round(y)
        if m.conv == op.name and m.fault == 'channel_off':
          y = torch.cat([torch.zeros_like(y[:, :1]), y[:, :-1]], dim=1)
        if s.kind == 'conv+maxpool':
          store(s.pool.dst, 0, F.max_pool2d(y, 3, 2), ch[s.pool.dst])
        else:
          store(op.dst, op.dst_channel_offset, y, op.cout if s.no_act else ch[op.dst])
      elif s.kind == 'maxpool':
        store(op.dst, op.dst_channel_offset, F.max_pool2d(t[op.src], 3, 2), ch[op.dst])
      else:
        y = _avgpool(t[op.src])
        if s.ci >= 0:
          y = torch.relu(y + self.convs[s.ci][1].view(1, -1, 1, 1))
        store(op.dst, op.dst_channel_offset, self._round(y), ch[op.dst])
    self.pooled = t['mixed10'].mean(dim=(2, 3))
    self.tensors = {k: v.permute(0, 2, 3, 1).contiguous().numpy() for k, v in t.items()}
    self.tensors['pooled'] = self.pooled.reshape(n, 1, 1, -1).numpy()
    return torch.softmax(self.pooled @ self.dk + self.db, dim=1).numpy()

  def debug_tensor(self, name: str, n: int) -> np.ndarray:
    return self.tensors[name][:n]      # KeyError for a tensor the engine does not materialise


def _images(n, shape, seed):
  g = torch.Generator().manual_seed(seed)
  return torch.randint(0, 255, (n,) + tuple(shape), dtype=torch.uint8, generator=g).numpy()


def smallest_side() -> int:
  """The smallest image side (height or width) for which every op of the graph has an output (modeling.out_hw)."""
  ops, _ = modeling.inception_v3_graph(7)

  def fits(side):
    hw = {'input': (side, side)}
    for o in ops:
      h, w = modeling.out_hw(o, *hw[o.src])
      if h < 1 or w < 1:
        return False
      hw[o.dst] = (h, w)
    return True

  return next(s for s in range(3, 400) if fits(s))


EDGE = (smallest_side(), smallest_side(), 16)     # 16 channels: stem patches of 9 x 16 = 144 -> stem_Kp 160; deep maps 1x1


def _check_emulated(shape, n, mutant=None, idx=None, seed=1):
  w = modeling.random_weights(shape[2], seed)
  blob = modeling.pack_weights(w)
  eng = Fp16Engine(blob, shape[2], mutant)
  imgs = _images(n, shape, seed)
  probs = eng.forward_host(imgs)
  chk = LayerChecker(lambda name: eng.debug_tensor(name, n), blob, imgs, probs, range(n) if idx is None else idx, Route())
  return chk.run(), eng, w, imgs, probs


# ---- CPU: the checker passes a correct fp16 engine and catches faulty ones -------------------------------------------------------

def test_smallest_geometry_is_75():
  assert EDGE[:2] == (75, 75)
  ops, _ = modeling.inception_v3_graph(16)
  hw = {'input': EDGE[:2]}
  for o in ops:
    hw[o.dst] = modeling.out_hw(o, *hw[o.src])
  assert hw['mixed10'] == (1, 1)


@pytest.mark.parametrize('shape', GEOMETRIES + [EDGE])
def test_checker_passes_emulated_fp16_engine(shape):
  chk, *_ = _check_emulated(shape, 2)
  chk.assert_ok(f'emulated fp16 engine {shape}')


MUTANTS = [
    Mutant('conv42 (mixed5_s1, merged 1x1 member) bias dropped', 'conv42', 'drop_bias'),
    Mutant('conv49 (mixed5[384:576]) bias dropped', 'conv49', 'drop_bias'),
    Mutant('conv17 (mixed1_d2, 3x3 same) tap (0, 0) dropped on the last output row', 'conv17', 'drop_tap'),
    Mutant('conv34 (mixed4[192:384], 7x1) last image computed from the previous image', 'conv34', 'prev_image'),
    Mutant('outputs truncated to fp16', None, 'truncate'),
    Mutant('conv42 written one channel off', 'conv42', 'channel_off'),
]

# The old end-to-end bar (test_cnn_gpu.py: stem 6e-3, blocks and branch tensors 2e-2 of scale, probabilities 5e-3 from the
# fp32 oracle) on the same mutants: True = the mutant passes it.
OLD_BAR_VERDICT = {
    'conv42 (mixed5_s1, merged 1x1 member) bias dropped': True,
    'conv49 (mixed5[384:576]) bias dropped': True,
    'conv17 (mixed1_d2, 3x3 same) tap (0, 0) dropped on the last output row': False,
    'conv34 (mixed4[192:384], 7x1) last image computed from the previous image': False,
    'outputs truncated to fp16': True,
    'conv42 written one channel off': False,
}


def test_mutant_layers_are_the_ones_named():
  ops, _ = modeling.inception_v3_graph(7)
  by_name = {o.name: o for o in ops if o.kind == 'conv'}
  assert (by_name['conv42'].dst, by_name['conv42'].src) == ('mixed5_s1', 'mixed4')
  assert (by_name['conv49'].dst, by_name['conv49'].dst_channel_offset) == ('mixed5', 384)
  assert (by_name['conv17'].dst, by_name['conv17'].same, by_name['conv17'].kh) == ('mixed1_d2', True, 3)
  assert (by_name['conv34'].dst, by_name['conv34'].dst_channel_offset, by_name['conv34'].kh) == ('mixed4', 192, 7)


@pytest.mark.parametrize('mutant', MUTANTS, ids=[m.fault + ('_' + m.conv if m.conv else '') for m in MUTANTS])
def test_checker_catches_mutant(mutant):
  chk, *_ = _check_emulated((100, 221, 7), 2, mutant)
  chk.print_report(mutant.name)
  assert chk.failures, f'{mutant.name}: not caught'
  first = chk.failures[0]
  print('first failure:', first)
  if mutant.conv:     # the checker points at the faulty layer, not at the block after it
    assert first.startswith(mutant.conv + ' '), first
  else:
    assert first.startswith('conv1 '), first


STEM_NAMES = ['s1', 's2', 'p1', 's4', 's5', 'p2']
BLOCKS = STEM_NAMES + [f'mixed{i}' for i in range(11)]
BRANCHES = ['mixed0_b5a', 'mixed0_d2', 'mixed3_d2', 'mixed4_s2', 'mixed4_d4', 'mixed8_b3', 'mixed9_t1', 'mixed9_d2']


def old_bar(eng, w, imgs, probs):
  """test_cnn_gpu.py's thresholds on the emulated engine: (passes, worst block error of scale, probability error)."""
  import cnn_oracle
  want_p, tensors, _ = cnn_oracle.ReferenceModel(w).forward(torch.from_numpy(imgs), return_tensors=True)
  worst, ok = 0.0, True
  for name in BLOCKS + BRANCHES:
    ref = tensors[name].permute(0, 2, 3, 1).numpy()
    err = float(np.abs(eng.debug_tensor(name, len(imgs)) - ref).max()) / max(float(np.abs(ref).max()), 1e-6)
    ok &= err < (6e-3 if name in STEM_NAMES else 2e-2)
    worst = max(worst, err)
  perr = float(np.abs(probs - want_p.numpy()).max())
  return ok and perr < 5e-3, worst, perr


def test_old_end_to_end_bar_misses_what_the_layer_checker_catches():
  _, eng, w, imgs, probs = _check_emulated((100, 221, 7), 2)
  assert old_bar(eng, w, imgs, probs)[0], 'the unmutated emulation must pass the old bar'
  got = {}
  for m in MUTANTS:
    _, eng, w, imgs, probs = _check_emulated((100, 221, 7), 2, m)
    ok, worst, perr = old_bar(eng, w, imgs, probs)
    print(f'{m.name:58s} old bar {"passes" if ok else "FAILS"}: worst block error {worst:.2g} of scale, probabilities {perr:.2g}')
    got[m.name] = ok
  assert got == OLD_BAR_VERDICT
  assert got['conv42 (mixed5_s1, merged 1x1 member) bias dropped'] and got['conv49 (mixed5[384:576]) bias dropped']


# ---- GPU: the CUDA engine, layer by layer ------------------------------------------------------------------------------------------

def _gpu_net(shape, max_batch, precision=0, seed=7):
  from deepvariant_b200 import call_variants as cv
  w = modeling.random_weights(shape[2], seed)
  return cv.GpuCnn(w, shape, device=0, max_batch=max_batch, precision=precision), modeling.pack_weights(w, precision)


def _check_gpu(net, blob, imgs, probs, idx, route, title, from_tensor=None):
  n = len(imgs)
  chk = LayerChecker(lambda name: net.debug_tensor(name, n), blob, imgs, probs, idx, route, from_tensor).run()
  chk.assert_ok(title)
  return chk


def _shape_id(shape):
  return 'x'.join(str(v) for v in shape)


@pytest.mark.gpu
@pytest.mark.parametrize('batch', ['n1', 'n3_after_n5'])
@pytest.mark.parametrize('shape', GEOMETRIES + [EDGE], ids=_shape_id)
def test_every_layer_matches_float64(shape, batch):
  """Default plan at every geometry make_examples builds the classifier for (WGS 7 channels, PacBio 100x147x10, the CLI
  default of 6 channels, WGS with diff_channels' 9, the DeepTrio height 140) and at the smallest image the graph accepts
  (16 channels).  One image alone; and three images (odd: the last CTA stream of conv_rows_kernel is short) in an engine
  of max_batch 5 that has just run five other images, so every buffer past the third image holds stale activations."""
  if batch == 'n1':
    net, blob = _gpu_net(shape, 1)
    imgs, idx = _images(1, shape, 40), [0]
  else:
    net, blob = _gpu_net(shape, 5)
    net.forward_host(_images(5, shape, 41))
    imgs, idx = _images(3, shape, 42), [0, 2]
  probs = net.forward_host(imgs)
  _check_gpu(net, blob, imgs, probs, idx, Route(), f'default plan {shape} {batch}')
  net.close()


@pytest.mark.gpu
@pytest.mark.parametrize('hw', [(EDGE[0] - 1, EDGE[1]), (EDGE[0], EDGE[1] - 1)], ids=['height', 'width'])
def test_one_pixel_below_the_smallest_image_is_refused(hw):
  from deepvariant_b200 import _lib, call_variants as cv
  with pytest.raises(_lib.DvbError) as e:
    cv.GpuCnn(modeling.random_weights(EDGE[2], 0), hw + (EDGE[2],), device=0, max_batch=1)
  assert e.value.status == 1, e.value     # DVB_ERR_INVALID_ARGUMENT


# route -> (environment, precision).  DVB_CNN_AVGPOOL_FLAT=1 (avgpool3x3s1_kernel) is the default, so the default plan covers it;
# the route below turns it off (pool3x3_kernel, the sliding form).
ROUTES = {
    'default': ({}, 0),
    'persistent': ({'DVB_CNN_PERSIST': '2'}, 0),
    'pair': ({'DVB_CNN_PERSIST': '2', 'DVB_CNN_PAIR': '1'}, 0),
    'halo_no_rows': ({'DVB_CNN_ROWS': '0'}, 0),
    'halo_rule2': ({'DVB_HALO_RULE': '2'}, 0),
    'stem_patch': ({'DVB_CNN_STEM_FUSED': '0'}, 0),
    'stem_rows': ({'DVB_CNN_STEM_ROWS': '1'}, 0),
    'no_merge': ({'DVB_CNN_MERGE_1X1': '0'}, 0),
    'unfused_pool': ({'DVB_CNN_FUSE_POOL': '0'}, 0),
    'pool_first': ({'DVB_CNN_POOL_AFTER_CONV': '0'}, 0),
    'sliding_avgpool': ({'DVB_CNN_AVGPOOL_FLAT': '0'}, 0),
    'precision1': ({}, 1),
}


def _plan(listing):
  lines = listing.splitlines()
  get = lambda tag: [l for l in lines if l.startswith(tag)]
  return {'stem': get('[stem]'), 'conv': get('[conv '), 'halo': get('[halo '), 'rows': get('[rows '), 'pool': get('[pool ')}


def _dst(line):
  return re.search(r' dst=(\S+)', line).group(1)


def _assert_engaged(route, plan, shape, precision):
  """The DVB_CNN_LIST plan shows that the route's kernels run (else the case would pass without testing them)."""
  stem = plan['stem'][0]
  steps = plan['conv'] + plan['halo'] + plan['rows']
  avg = [l for l in plan['pool'] if '] avg ' in l]
  assert len(avg) == 9 and len(plan['pool']) == 9 + 4 - (1 if any('pool=1' in l for l in plan['rows']) else 0), plan['pool']
  if route == 'default':
    assert stem == ('[stem] fused' if shape[2] == 7 else '[stem] patch')
    assert any(_dst(l) == 'p1' and 'pool=1' in l for l in plan['rows'])
    assert all('kernel=avgpool3x3s1' in l and 'bias=1' in l for l in avg)
    assert len(steps) + (stem != '[stem] patch') < 94                     # merged 1x1 groups
  elif route == 'persistent':
    assert sum('persist=1 pair=0' in l for l in plan['conv']) >= 20
  elif route == 'pair':
    assert sum('pair=1' in l for l in plan['conv']) >= 20
  elif route == 'halo_no_rows':
    assert not plan['rows']
    assert {'s2', 's3'} <= {_dst(l) for l in steps}
  elif route == 'halo_rule2':
    assert plan['halo']
  elif route == 'stem_patch':
    assert stem == '[stem] patch' and any(_dst(l) == 's1' for l in plan['conv'])
  elif route == 'stem_rows':
    assert stem == '[stem] rows'
  elif route == 'no_merge':
    assert len(steps) + (stem != '[stem] patch') == 94
  elif route == 'unfused_pool':
    assert any(_dst(l) == 's3' and 'pool=0' in l for l in plan['rows'])
  elif route == 'pool_first':
    assert all('bias=0' in l and _dst(l).endswith('_ap') for l in avg)
  elif route == 'sliding_avgpool':
    assert all('kernel=pool3x3' in l for l in avg)
  elif route == 'precision1':
    assert stem == '[stem] patch' and not plan['rows'] and not plan['halo']
    assert not any('persist=1' in l for l in plan['conv']) and all('kernel=pool3x3' in l for l in plan['pool'])
  else:
    raise AssertionError(route)


@pytest.mark.gpu
@pytest.mark.parametrize('geometry', ['wgs', 'other'])
@pytest.mark.parametrize('route', list(ROUTES))
def test_every_layer_matches_float64_on_each_kernel_route(monkeypatch, capfd, route, geometry):
  """Each kernel route at WGS and at one other geometry (100x147x10; 140x221x7 for the stem routes, which need 7 channels),
  three images, the first and the last checked."""
  env, precision = ROUTES[route]
  shape = (100, 221, 7) if geometry == 'wgs' else (140, 221, 7) if route.startswith('stem') else (100, 147, 10)
  monkeypatch.setenv('DVB_CNN_LIST', '1')
  for k, v in env.items():
    monkeypatch.setenv(k, v)
  capfd.readouterr()
  net, blob = _gpu_net(shape, 3, precision, seed=8)
  plan = _plan(capfd.readouterr().err)
  print('\n'.join(sum(plan.values(), [])))
  _assert_engaged(route, plan, shape, precision)
  imgs = _images(3, shape, 43)
  probs = net.forward_host(imgs)
  r = Route(precision, pool_after_conv=env.get('DVB_CNN_POOL_AFTER_CONV', '1') != '0',
            fused_pool=precision == 0 and env.get('DVB_CNN_ROWS', '1') != '0' and env.get('DVB_CNN_FUSE_POOL', '1') != '0')
  _check_gpu(net, blob, imgs, probs, [0, 2], r, f'{route} {shape}')
  net.close()


def _tile_images(line, t, n):
  """Images the M tile of persistent-kernel tile t (t = nb * m_tiles + m) covers, from a [conv] plan line."""
  f = {k: v for k, v in re.findall(r'(\w+)=(\S+)', line)}
  m = t % int(f['m_tiles'])
  H, W = (int(v) for v in f['out'].split('x'))
  if f['flat'] == '1':
    p0 = 128 * m
    return set(range(p0 // (H * W), min(p0 + 127, n * H * W - 1) // (H * W) + 1))
  Wt, Ht, Nt = (int(v) for v in f['box'].split('x'))
  tn = m // (-(-W // Wt) * -(-H // Ht))
  return set(range(tn * Nt, min(n, tn * Nt + Nt)))


@pytest.mark.gpu
def test_persistent_kernel_later_passes_match_float64(monkeypatch, capfd):
  """DVB_CNN_PERSIST=2 at 256 WGS images: conv_gemm_persistent_kernel CTAs take tiles b, b + G, b + 2G, ... (G = CTAs), so the
  TMA ring runs across tiles and the two TMEM accumulators alternate.  The layers from mixed0 on are checked on the first and
  last image and on the images of the tiles CTA 0 takes on its second and third pass through mixed0's merged 1x1 GEMM."""
  shape, n = (100, 221, 7), 256
  monkeypatch.setenv('DVB_CNN_LIST', '1')
  monkeypatch.setenv('DVB_CNN_PERSIST', '2')
  capfd.readouterr()
  net, blob = _gpu_net(shape, n, seed=9)
  plan = _plan(capfd.readouterr().err)
  num_sms = torch.cuda.get_device_properties(0).multi_processor_count
  passes = {}
  for l in plan['conv']:
    if 'persist=1' in l and _dst(l) not in passes:    # the first GEMM writing a tensor: for mixed0, its merged 1x1 group
      f = dict(re.findall(r'(\w+)=(\S+)', l))
      total = int(f['m_tiles']) * int(f['n_blocks'])
      passes[_dst(l)] = (-(-total // min(total, num_sms)), min(total, num_sms), l)
  print('passes per CTA:', {k: v[0] for k, v in passes.items()})
  n_pass, G, line = passes['mixed0']
  assert n_pass >= 3 and 'flat=1' in line, line
  idx = sorted({0, n - 1} | _tile_images(line, G, n) | _tile_images(line, 2 * G, n))
  assert len(idx) >= 4 and any(0 < i < n - 1 for i in idx), idx
  imgs = _images(n, shape, 44)
  probs = net.forward_host(imgs)
  _check_gpu(net, blob, imgs, probs, idx, Route(), f'persistent, {n} images, passes {n_pass}', from_tensor='p2')
  net.close()
