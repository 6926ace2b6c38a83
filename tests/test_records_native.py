"""call_variants record I/O in C++ (csrc/dvb_records.cu; SURVEY 8(a) rows a16 / a17) against the Python restatements
(tfrecord.read_records + protos.parse_tf_example; call_variants.round_gls + create_cvo) that the reference's golden
CallVariantsOutput file pins (tests/test_golden.py).  CPU-only: host code of libdvb.so."""
import ctypes as C
import gzip
import os
import struct

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from deepvariant_b200 import _lib, call_variants as cv, protos, records, tfrecord

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _example(image: bytes, variant: bytes, alt: bytes, shape=(2, 3, 1), extra=True) -> bytes:
  feats = {'image/encoded': ('bytes', [image]), 'variant/encoded': ('bytes', [variant]), 'alt_allele_indices/encoded': ('bytes', [alt]),
           'image/shape': ('int64', list(shape))}
  if extra:
    feats.update({'locus': ('bytes', [b'chr1:1-2']), 'variant_type': ('int64', [1]), 'sequencing_type': ('int64', [0])})
  return protos.encode_tf_example(feats)


def _call(name: bytes, info=()) -> bytes:
  """A VariantCall (variants.proto): call_set_name = 9, genotype = 7, info = 2 (map<string, ListValue>)."""
  out = b''
  for key, val in info:
    out += protos.f_bytes(2, protos.f_bytes(1, key) + protos.f_bytes(2, protos.f_bytes(1, protos.f_bytes(3, val))))
  return out + protos.f_bytes(7, protos.packed_varints([1, 1])) + protos.f_bytes(9, name)


def _variant(i: int) -> bytes:
  base = protos.Variant(reference_name='chr20', start=100 + i, end=101 + i, reference_bases='A', alternate_bases=['C']).serialize()
  return base + protos.f_bytes(11, _call(b's'))


def _write_shards(tmp_path, sizes, image_bytes=6, kinds=None):
  """Shards with the given record counts; kinds[i] in {'gz', 'plain', 'multi'} ('multi' = several gzip members)."""
  rng = np.random.default_rng(7)
  paths, content = [], []
  for i, n in enumerate(sizes):
    kind = (kinds or ['gz'] * len(sizes))[i]
    path = str(tmp_path / f'ex-{i:05d}-of-{len(sizes):05d}.tfrecord{"" if kind == "plain" else ".gz"}')
    recs = []
    for j in range(n):
      recs.append((rng.integers(0, 256, image_bytes, dtype=np.uint8).tobytes(), _variant(100 * i + j), bytes([8, j % 3])))
    if kind == 'multi':
      with open(path, 'wb') as f:
        for k in range(0, max(n, 1), 2):   # two records per gzip member
          raw = b''
          for img, v, a in recs[k:k + 2]:
            ex = _example(img, v, a)
            hdr = struct.pack('<Q', len(ex))
            raw += hdr + struct.pack('<I', tfrecord.masked_crc32c(hdr)) + ex + struct.pack('<I', tfrecord.masked_crc32c(ex))
          f.write(gzip.compress(raw))
    else:
      with tfrecord.Writer(path) as w:
        for img, v, a in recs:
          w.write(_example(img, v, a))
    paths.append(path)
    content.append(recs)
  return paths, content


def _drain(reader, image_bytes, batch):
  out = []
  buf = np.zeros((batch, image_bytes), dtype=np.uint8)
  while True:
    meta = reader.next_into(buf)
    if meta is None:
      return out
    out += list(zip([buf[i].tobytes() for i in range(meta.n)], meta.variants(), meta.alt_allele_indices()))


def test_crc32c_instruction_equals_table_walk():
  lib = _lib.lib()
  rng = np.random.default_rng(0)
  data = rng.integers(0, 256, 70000, dtype=np.uint8).tobytes()
  assert lib.dvb_crc32c(b'123456789', 9) == lib.dvb_crc32c_portable(b'123456789', 9) == 0xE3069283   # the CRC-32C check value
  for off, n in [(0, 0), (0, 1), (1, 7), (3, 8), (5, 64), (2, 1000), (7, 65535), (0, 70000)]:
    chunk = data[off:off + n]
    assert lib.dvb_crc32c(chunk, len(chunk)) == lib.dvb_crc32c_portable(chunk, len(chunk))


def test_interleave_order_known_answers():
  assert records.interleave_order([3, 1, 2], 2) == [(0, 0), (1, 0), (0, 1), (0, 2), (2, 0), (2, 1)]
  assert records.interleave_order([2, 2], 1) == [(0, 0), (0, 1), (1, 0), (1, 1)]
  assert records.interleave_order([2, 0, 1], 32) == [(0, 0), (2, 0), (0, 1)]
  assert records.interleave_order([], 4) == []


@pytest.mark.parametrize('cycle_length,threads,batch', [(2, 1, 3), (32, 4, 5), (3, 2, 1000), (1, 3, 4)])
def test_reader_order_and_content_on_ragged_shards(tmp_path, cycle_length, threads, batch):
  sizes = [5, 0, 9, 1, 4, 7]
  paths, content = _write_shards(tmp_path, sizes, kinds=['gz', 'gz', 'multi', 'plain', 'gz', 'multi'])
  with records.NativeExamplesReader(paths, threads=threads, cycle_length=cycle_length) as r:
    shape, nbytes = r.shape()
    assert shape == [2, 3, 1] and nbytes == 6
    got = _drain(r, 6, batch)
    assert r.next_into(np.zeros((2, 6), dtype=np.uint8)) is None   # stays at the end
  want = [content[s][k] for s, k in records.interleave_order(sizes, cycle_length)]
  assert got == want
  assert len(got) == sum(sizes)


def test_reader_without_records_and_without_files(tmp_path):
  paths, _ = _write_shards(tmp_path, [0, 0])
  with records.NativeExamplesReader(paths) as r:
    assert r.shape() == ([0, 0, 0], 0)
    assert r.next_into(np.zeros((4, 6), dtype=np.uint8)) is None
  with records.NativeExamplesReader([]) as r:
    assert r.shape() == ([0, 0, 0], 0)
  with pytest.raises(_lib.DvbError, match='cannot open'):
    records.NativeExamplesReader([str(tmp_path / 'missing.gz')])


def test_reader_errors(tmp_path):
  paths, _ = _write_shards(tmp_path, [3], image_bytes=4000)
  buf = np.zeros((8, 4000), dtype=np.uint8)
  # wrong image size
  with records.NativeExamplesReader(paths) as r:
    with pytest.raises(_lib.DvbError, match='image/encoded has 4000 bytes'):
      r.next_into(np.zeros((8, 6), dtype=np.uint8))
  # truncated gzip stream
  blob = open(paths[0], 'rb').read()
  bad = str(tmp_path / 'trunc.tfrecord.gz')
  open(bad, 'wb').write(blob[:len(blob) // 2])
  with records.NativeExamplesReader([bad]) as r:
    with pytest.raises(_lib.DvbError, match='truncated|corrupt'):
      while r.next_into(buf) is not None:
        pass
  # a flipped payload byte: caught by the record CRC, accepted (as garbage) without verification
  raw = bytearray(gzip.decompress(blob))
  raw[12 + 200] ^= 0x40
  bad = str(tmp_path / 'flip.tfrecord')
  open(bad, 'wb').write(bytes(raw))
  with records.NativeExamplesReader([bad]) as r:
    with pytest.raises(_lib.DvbError, match='corrupted record data'):
      r.next_into(buf)
  # truncated in the middle of a record (plain file)
  bad = str(tmp_path / 'cut.tfrecord')
  open(bad, 'wb').write(bytes(gzip.decompress(blob)[:-7]))
  with records.NativeExamplesReader([bad]) as r:
    with pytest.raises(_lib.DvbError, match='truncated TFRecord'):
      while r.next_into(buf) is not None:
        pass
  # a record without variant/encoded; one with two image values
  for feats, msg in [({'image/encoded': ('bytes', [b'x' * 6]), 'alt_allele_indices/encoded': ('bytes', [b''])}, 'variant/encoded'),
                     ({'image/encoded': ('bytes', [b'x' * 6, b'y' * 6]), 'variant/encoded': ('bytes', [b'v']),
                       'alt_allele_indices/encoded': ('bytes', [b''])}, 'image/encoded')]:
    bad = str(tmp_path / 'feat.tfrecord.gz')
    with tfrecord.Writer(bad) as w:
      w.write(protos.encode_tf_example(feats))
    with records.NativeExamplesReader([bad]) as r:
      with pytest.raises(_lib.DvbError, match=msg):
        r.next_into(np.zeros((2, 6), dtype=np.uint8))


def test_reader_on_the_reference_golden_examples():
  path = os.path.join(GOLDEN, 'golden.calling_examples.tfrecord.gz')
  want = [protos.parse_tf_example(r) for r in tfrecord.read_records(path)]
  with records.NativeExamplesReader([path]) as r:
    shape, nbytes = r.shape()
    assert shape == [int(x) for x in want[0]['image/shape'][1]] and nbytes == shape[0] * shape[1] * shape[2]
    got = _drain(r, nbytes, 32)
  assert len(got) == len(want) == 84
  for (img, v, a), ex in zip(got, want):
    assert img == ex['image/encoded'][1][0] and v == ex['variant/encoded'][1][0] and a == ex['alt_allele_indices/encoded'][1][0]


def _native_round(gls, precision=10):
  a = (C.c_double * 3)(*gls)
  out = (C.c_double * 3)()
  _lib.check(_lib.lib().dvb_debug_round_gls(a, precision, out))
  return list(out)


def test_round_gls_known_answers():
  for gls in ([1.0, 0.0, 0.0], [0.5, 0.5, 0.0], [1 / 3, 1 / 3, 1 / 3], [0.25, 0.25, 0.5], [0.12345678905, 0.87654321095, 0.0],
              [0.00000000005, 0.99999999995, 0.0], [0.99999994, 2e-8, 4e-8], [0.3333333432674408, 0.3333333432674408, 0.3333333134651184]):
    assert _native_round(gls) == cv.round_gls(gls, 10), gls
    assert _native_round(gls, -1) == cv.round_gls(gls, None)
    assert _native_round(gls, 3) == cv.round_gls(gls, 3)
  with pytest.raises(_lib.DvbError, match='do not sum to one'):
    _native_round([0.5, 0.5, 0.1])


@settings(max_examples=400, deadline=None)
@given(st.lists(st.floats(-30, 30, width=32), min_size=3, max_size=3), st.integers(0, 12))
def test_round_gls_equals_python_on_float32_softmax_outputs(logits, precision):
  """The probabilities the classifier hands over are float32 softmax outputs widened to float64."""
  z = np.array(logits, dtype=np.float32)
  e = np.exp(z - z.max())
  gls = [float(x) for x in (e / e.sum()).astype(np.float32)]
  assert _native_round(gls, precision) == cv.round_gls(gls, precision)


@pytest.mark.parametrize('suffix', ['.tfrecord.gz', '.tfrecord'])
def test_cvo_writer_equals_python_records(tmp_path, suffix):
  rng = np.random.default_rng(3)
  n = 500
  logits = rng.normal(0, 4, (n, 3)).astype(np.float32)
  e = np.exp(logits - logits.max(1, keepdims=True))
  probs = (e / e.sum(1, keepdims=True)).astype(np.float32)
  probs[0] = [1, 0, 0]
  probs[1] = [0.5, 0.5, 0]
  variants = [_variant(i) for i in range(n)]
  # a variant that already carries a MID entry and other info, and one with two calls
  base = protos.Variant(reference_name='chr1', start=5, end=6, reference_bases='G', alternate_bases=['T', 'GA']).serialize()
  variants[2] = base + protos.f_bytes(11, _call(b'a', [(b'DP', b'7'), (b'MID', b'old'), (b'AD', b'3')])) + protos.f_bytes(11, _call(b'b', [(b'MID', b'keep')]))
  variants[3] = protos.f_bytes(11, _call(b'first')) + base   # fields in non-canonical order stay where they are
  alts = [bytes([8, i % 2]) if i % 5 else b'' for i in range(n)]
  path = str(tmp_path / f'cvo{suffix}')
  w = records.NativeCvoWriter(path)
  for a in range(0, n, 128):   # several batches
    b = min(n, a + 128)
    w.write_batch(records.BatchMeta.from_lists(variants[a:b], alts[a:b]), probs[a:b])
  assert w.close() == n
  got = list(tfrecord.read_records(path, check_crc=True))
  want = [cv.create_cvo(variants[i], cv.round_gls(probs[i].astype(np.float64).tolist(), 10), alts[i]) for i in range(n)]
  assert got == want
  variant2 = protos.parse_call_variants_output(got[2])[0]
  assert variant2.count(b'MID') == 2 and b'old' not in variant2 and b'keep' in variant2 and variant2.count(b'deepvariant') == 1


def test_cvo_writer_errors(tmp_path):
  meta = records.BatchMeta.from_lists([_variant(0)], [b''])
  w = records.NativeCvoWriter(str(tmp_path / 'a.gz'))
  w.write_batch(meta, np.array([[0.5, 0.5, 0.5]], dtype=np.float32))
  with pytest.raises(_lib.DvbError, match='do not sum to one'):
    w.close()
  no_calls = protos.Variant(reference_name='chr1', start=1, end=2, reference_bases='A', alternate_bases=['C']).serialize()
  w = records.NativeCvoWriter(str(tmp_path / 'b.gz'))
  w.write_batch(records.BatchMeta.from_lists([no_calls], [b'']), np.array([[1, 0, 0]], dtype=np.float32))
  with pytest.raises(_lib.DvbError, match='no calls'):
    w.close()
  with pytest.raises(_lib.DvbError, match='cannot create'):
    records.NativeCvoWriter(str(tmp_path / 'nodir' / 'c.gz'))
  w = records.NativeCvoWriter(str(tmp_path / 'd.gz'))
  with pytest.raises(ValueError):
    w.write_batch(meta, np.zeros((2, 3), dtype=np.float32))
  assert w.close() == 0
  assert list(tfrecord.read_records(str(tmp_path / 'd.gz'))) == []


@settings(max_examples=400, deadline=None)
@given(st.floats(0, 1), st.floats(0, 1), st.integers(0, 12))
def test_round_gls_equals_python_on_arbitrary_doubles(a, b, precision):
  gls = [a * (1 - b), (1 - a) * (1 - b), b]
  if abs(sum(gls) - 1) > 1e-7:
    return
  assert _native_round(gls, precision) == cv.round_gls(gls, precision)


def test_reader_many_shards_many_threads_repeatedly(tmp_path):
  """Scheduling stress: 40 small shards, more threads than cores, queues shorter than the shards."""
  sizes = [(7 * i) % 23 for i in range(40)]
  paths, content = _write_shards(tmp_path, sizes, image_bytes=64)
  want = [content[s][k] for s, k in records.interleave_order(sizes, 32)]
  for rep in range(8):
    with records.NativeExamplesReader(paths, threads=1 + 3 * rep, cycle_length=32, verify_crc=bool(rep % 2)) as r:
      assert _drain(r, 64, 1 + 17 * rep) == want
  # closing a reader that was never drained must not hang
  r = records.NativeExamplesReader(paths, threads=8)
  r.next_into(np.zeros((3, 64), dtype=np.uint8))
  r.close()
