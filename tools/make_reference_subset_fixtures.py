"""Builds the fixtures under tests/golden/ that the tests comparing with DeepVariant's own testdata (deepvariant/testdata of the
original project) read instead of it:

  golden.calling_candidates.tfrecord.gz          copied as is (78 DeepVariantCalls of chr20:10,000,000-10,010,000)
  golden.calling_examples.tfrecord.gz            copied as is (84 examples of the same region)
  golden.calling_examples.shard_keys.json        (start, alt allele indices) of the examples of each of its three --task shards
  golden.alt_aligned_pileup.digests.json         per example of golden.alt_aligned_pileup_{diff_channels,rows}_examples:
                                                 (start, alt allele indices) and the SHA-256 of its image (image_digest)
  NA12878_S1.chr20.10_10p1mb.window.bam(.bai)    the records of input/NA12878_S1.chr20.10_10p1mb.bam that start before
                                                 chr20:10,011,000, byte for byte, in fresh BGZF blocks, and its index
  NA12878_S1.chr20.10_10p1mb.first_container.cram   its CRAM's file definition, header container, first data container
                                                 (10,000 records from chr20:9,999,912) and EOF container
  reads_head.<name>.bam                          the first records of three of its BAMs, byte for byte, in fresh BGZF blocks
  test_pacbio.chr20_9060000_9065000.bam          the records of input/test_pacbio.chr20_100kbp_at_9mb.bam overlapping
                                                 chr20:9,060,000-9,065,000, byte for byte
  golden.pacbio_variants.chr20_9060000_9065000.json  the variants of golden.pacbio_examples in that window (canonical_call fields)
  test_pacbio.chr20_9074999_9099999.bam          its records overlapping chr20:9,069,999-9,104,999 (the partition 9,074,999-9,099,999
                                                 and its padding), byte for byte
  golden.pacbio_examples.chr20_9074999_9099999.json  per example of golden.pacbio_examples in that partition: (start, alt allele
                                                 indices) and check_pacbio_end_to_end.channel_summary of its image
  grch38.chr20_9030000_9135000.fa.gz             chr20 of input/grch38.chr20_and_21_10M.fa.gz, N outside 9,030,000-9,135,000
The NA12878 reads lie in chr20:9,990,000-10,020,000, where tests/golden/quickstart.chr20_10mb.fa.gz holds the reference bases.

Usage:  python tools/make_reference_subset_fixtures.py <deepvariant/testdata directory>"""
import gzip
import json
import os
import shutil
import struct
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepvariant_b200 import protos, tfrecord  # noqa: E402
from deepvariant_b200.bgzf_tabix import bgzf_member, reg2bin  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from check_alt_aligned_wgs_golden import image_digest  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
# (BAM, records kept): long-read records are about 10 kB each
BAM_HEADS = (('NA12878_S1.chr20.10_10p1mb.bam', 400), ('test_pacbio.chr20_100kbp_at_9mb.bam', 16),
             ('HG002.hifi.hg37.phased.chr20.1_1000000.bam', 16))
WINDOW_END = 10_011_000
PACBIO_WINDOW = ('chr20', 9_060_000, 9_065_000)      # a 5-kb piece of the 100 kb of golden.pacbio_examples
PACBIO_PARTITION = ('chr20', 9_074_999, 9_099_999)   # one of its 25-kb partitions (the smallest whose padded reads fit in 1 MB)
PACBIO_PADDING = 5_000                                # 20 % of the partition, the padding candidates are called over
PACBIO_FASTA = ('chr20', 9_030_000, 9_135_000)       # reference bases kept, enough for the longest reads of both


def example_key(e: dict) -> list:
  return [protos.parse_variant(e['variant/encoded'][1][0]).start, list(protos.parse_alt_allele_indices(e['alt_allele_indices/encoded'][1][0]))]


def _write_bgzf(dst: str, payload: bytes, block: int = 0xff00) -> list:
  """Writes payload in BGZF blocks of `block` bytes; returns the file offset of every block, then that of the EOF block."""
  offsets = [0]
  with open(dst, 'wb') as f:
    for i in range(0, len(payload), block):
      offsets.append(offsets[-1] + f.write(bgzf_member(payload[i:i + block], 9)))
    f.write(bgzf_member(b''))
  return offsets


def _records(data: bytes):
  """(ref_id, start, end, offset, next offset) of every record of an uncompressed BAM, and the number of references."""
  p = 8 + struct.unpack_from('<i', data, 4)[0]
  n_ref = struct.unpack_from('<i', data, p)[0]
  p += 4
  for _ in range(n_ref):
    p += 4 + struct.unpack_from('<i', data, p)[0] + 4
  out = []
  while p < len(data):
    size = struct.unpack_from('<i', data, p)[0]
    ref_id, pos, l_name = struct.unpack_from('<iiB', data, p + 4)
    n_cigar = struct.unpack_from('<H', data, p + 16)[0]
    ops = struct.unpack_from(f'<{n_cigar}I', data, p + 36 + l_name)
    out.append((ref_id, pos, pos + sum(c >> 4 for c in ops if (c & 0xf) in (0, 2, 3, 7, 8)), p, p + 4 + size))
    p += 4 + size
  return out, n_ref


def write_bai(dst: str, payload: bytes, offsets: list, block: int = 0xff00) -> None:
  """The .bai (SAM spec 5.2) of a BAM that _write_bgzf wrote from payload: one chunk per record in its bin, and the linear index."""
  def voffset(u):
    return offsets[u // block] << 16 | u % block if u < len(payload) else offsets[-1] << 16
  records, n_ref = _records(payload)
  bins = [dict() for _ in range(n_ref)]
  linear = [dict() for _ in range(n_ref)]
  for ref_id, pos, end, u0, u1 in records:
    if ref_id < 0:
      continue
    chunks = bins[ref_id].setdefault(reg2bin(pos, max(end, pos + 1)), [])
    if chunks and chunks[-1][1] == voffset(u0):
      chunks[-1][1] = voffset(u1)
    else:
      chunks.append([voffset(u0), voffset(u1)])
    for w in range(pos >> 14, (max(end, pos + 1) - 1 >> 14) + 1):
      linear[ref_id].setdefault(w, voffset(u0))
  out = bytearray(b'BAI\1' + struct.pack('<i', n_ref))
  for r in range(n_ref):
    out += struct.pack('<i', len(bins[r]))
    for b, chunks in sorted(bins[r].items()):
      out += struct.pack('<Ii', b, len(chunks)) + b''.join(struct.pack('<QQ', *c) for c in chunks)
    n_intv = max(linear[r]) + 1 if linear[r] else 0
    ioff, last = [], 0
    for w in range(n_intv):
      last = linear[r].get(w, last)
      ioff.append(last)
    out += struct.pack('<i', n_intv) + struct.pack(f'<{n_intv}Q', *ioff)
  with open(dst, 'wb') as f:
    f.write(bytes(out))


def bam_records(src: str, keep):
  """The header and the records for which keep(index, ref_id, start, end) holds, unchanged; returns (bytes, record count)."""
  with gzip.open(src, 'rb') as f:
    data = f.read()
  records, _ = _records(data)
  kept = [data[u0:u1] for i, (ref_id, pos, end, u0, u1) in enumerate(records) if keep(i, ref_id, pos, end)]
  return data[:records[0][3] if records else len(data)] + b''.join(kept), len(kept)


def cram_first_container(src: str, dst: str) -> None:
  """CRAM 3.0: file definition, header container, first data container, EOF container (the last 38 bytes)."""
  with open(src, 'rb') as f:
    b = f.read()
  assert b[:4] == b'CRAM' and b[4] == 3
  p, ends = 26, []
  for _ in range(2):                        # container header: int32 length, then ITF8 / LTF8 fields ending in a CRC32
    length = struct.unpack_from('<i', b, p)[0]
    q, itf8s = p + 4, 0
    while itf8s < 4:                        # ref id, start, span, record count
      q += _itf8_len(b[q]); itf8s += 1
    q += _ltf8_len(b[q]); q += _ltf8_len(b[q])   # record counter, bases
    q += _itf8_len(b[q])                    # blocks
    n_land = _itf8(b, q)
    q += _itf8_len(b[q])
    for _ in range(n_land):
      q += _itf8_len(b[q])
    p = q + 4 + length
    ends.append(p)
  with open(dst, 'wb') as f:
    f.write(b[:ends[1]] + b[-38:])


def _itf8_len(c: int) -> int:
  return 1 if c < 0x80 else 2 if c < 0xc0 else 3 if c < 0xe0 else 4 if c < 0xf0 else 5


def _ltf8_len(c: int) -> int:
  n = 0
  while n < 8 and c & (0x80 >> n):
    n += 1
  return n + 1


def _itf8(b: bytes, p: int) -> int:
  n = _itf8_len(b[p])
  assert n == 1, 'small ITF8 expected'
  return b[p]


def masked_fasta(src: str, dst: str, contig: str, lo: int, hi: int) -> None:
  """A gzip FASTA of one contig, its bases in [lo, hi) and N elsewhere, with its .fai."""
  from deepvariant_b200 import fasta
  ref = fasta.IndexedFastaReader(src)
  n = ref.n_bases(contig)
  seq = 'N' * lo + ref.query(contig, lo, hi) + 'N' * (n - hi)
  with gzip.GzipFile(dst, 'wb', 9, mtime=0) as f:
    f.write(f'>{contig}\n'.encode())
    for i in range(0, n, 1 << 20):
      chunk = seq[i:i + (1 << 20)]
      f.write(''.join(chunk[j:j + 50] + '\n' for j in range(0, len(chunk), 50)).encode())
  with open(dst + '.fai', 'w') as f:
    f.write(f'{contig}\t{n}\t{len(contig) + 2}\t50\t51\n')


def pacbio_fixtures(td: str) -> None:
  """Reads overlapping PACBIO_WINDOW and the golden variants in it; reads overlapping the padded PACBIO_PARTITION and the
  channel summaries of its golden examples; the reference around both."""
  import check_candidates_golden as ck
  import check_pacbio_end_to_end as e2e
  from deepvariant_b200 import bam
  src = os.path.join(td, 'input', 'test_pacbio.chr20_100kbp_at_9mb.bam')
  rid = bam.NativeBamTable(src).references.index('chr20')
  spans = []

  def cut(name, a, b):
    def keep(i, r, pos, end):
      if r == rid and pos < b and end > a:
        spans.append((pos, end))
        return True
      return False
    payload, n = bam_records(src, keep)
    _write_bgzf(os.path.join(OUT, name), payload)
    return n

  contig, a, b = PACBIO_WINDOW
  n = cut('test_pacbio.chr20_9060000_9065000.bam', a, b)
  gold = ck.pacbio_golden_variants(os.path.join(td, 'golden.pacbio_examples.tfrecord.gz'))
  window = [c for c in gold.values() if c['contig'] == contig and a <= c['start'] < b]
  with open(os.path.join(OUT, 'golden.pacbio_variants.chr20_9060000_9065000.json'), 'w') as f:
    json.dump(window, f, indent=0)
  print('pacbio window', n, 'reads,', len(window), 'golden variants')
  contig, a, b = PACBIO_PARTITION
  n = cut('test_pacbio.chr20_9074999_9099999.bam', a - PACBIO_PADDING, b + PACBIO_PADDING)
  examples = [x for x in e2e.golden_summaries(os.path.join(td, 'golden.pacbio_examples.tfrecord.gz')) if a <= x[0] < b]
  with open(os.path.join(OUT, 'golden.pacbio_examples.chr20_9074999_9099999.json'), 'w') as f:
    json.dump(examples, f)
  print('pacbio partition', n, 'reads,', len(examples), 'golden examples')
  contig, lo, hi = PACBIO_FASTA
  assert lo <= min(p for p, _ in spans) and max(e for _, e in spans) <= hi, 'the FASTA fixture does not cover the reads'
  masked_fasta(os.path.join(td, 'input', 'grch38.chr20_and_21_10M.fa.gz'), os.path.join(OUT, 'grch38.chr20_9030000_9135000.fa.gz'), contig, lo, hi)


def main(td: str) -> None:
  inp = os.path.join(td, 'input')
  for name in ('golden.calling_candidates.tfrecord.gz', 'golden.calling_examples.tfrecord.gz'):
    shutil.copyfile(os.path.join(td, name), os.path.join(OUT, name))
  shards = [[example_key(protos.parse_tf_example(r)) for r in tfrecord.read_records(os.path.join(td, f'golden.calling_examples.tfrecord.gz-0000{i}-of-00003'))]
            for i in range(3)]
  with open(os.path.join(OUT, 'golden.calling_examples.shard_keys.json'), 'w') as f:
    json.dump(shards, f)
  digests = {}
  for layout in ('diff_channels', 'rows'):
    rows = []
    for r in tfrecord.read_records(os.path.join(td, f'golden.alt_aligned_pileup_{layout}_examples.tfrecord.gz')):
      e = protos.parse_tf_example(r)
      rows.append(example_key(e) + [image_digest(e['image/encoded'][1][0], e['image/shape'][1])])
    digests[layout] = rows
  with open(os.path.join(OUT, 'golden.alt_aligned_pileup.digests.json'), 'w') as f:
    json.dump(digests, f)
  payload, n = bam_records(os.path.join(inp, 'NA12878_S1.chr20.10_10p1mb.bam'), lambda i, rid, pos, end: pos < WINDOW_END)
  window = os.path.join(OUT, 'NA12878_S1.chr20.10_10p1mb.window.bam')
  write_bai(window + '.bai', payload, _write_bgzf(window, payload))
  print('window BAM', n, 'records')
  cram_first_container(os.path.join(inp, 'NA12878_S1.chr20.10_10p1mb.cram'), os.path.join(OUT, 'NA12878_S1.chr20.10_10p1mb.first_container.cram'))
  for name, k in BAM_HEADS:
    payload, n = bam_records(os.path.join(inp, name), lambda i, rid, pos, end, k=k: i < k)
    _write_bgzf(os.path.join(OUT, 'reads_head.' + name), payload)
    print(name, n, 'records')
  pacbio_fixtures(td)


if __name__ == '__main__':
  main(sys.argv[1])
