"""Native BAM decoder (csrc/dvb_bam.cu, SURVEY 8(f) next row #1) against the pure-Python reader and hand-built files.
CPU-only (host code of libdvb.so; no compute kernel is called)."""
import os
import struct
import zlib

import numpy as np
import pytest

from deepvariant_b200 import _lib, bam

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _bgzf(payload: bytes, block=30000) -> bytes:
  """BGZF container: gzip members with the 'BC' extra field, then the 28-byte EOF block."""
  out = bytearray()
  chunks = [payload[i:i + block] for i in range(0, len(payload), block)] + [b'']
  for ch in chunks:
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = co.compress(ch) + co.flush()
    bsize = len(body) + 12 + 6 + 8
    out += struct.pack('<4BI2BH2BHH', 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, ord('B'), ord('C'), 2, bsize - 1)
    out += body + struct.pack('<II', zlib.crc32(ch) & 0xffffffff, len(ch))
  return bytes(out)


_CODES = {c: i for i, c in enumerate('=ACMGRSVTWYHKDBN')}


def _record(ref_id, pos, name, mapq, flag, cigar, seq, qual, next_ref=-1, next_pos=-1, tlen=0, aux=b''):
  packed = bytearray((len(seq) + 1) // 2)
  for i, ch in enumerate(seq):
    packed[i >> 1] |= _CODES[ch] << (4 if i % 2 == 0 else 0)
  body = struct.pack('<iiBBHHHiiii', ref_id, pos, len(name) + 1, mapq, 0, len(cigar), flag, len(seq), next_ref, next_pos, tlen)
  body += name.encode() + b'\0' + b''.join(struct.pack('<I', (ln << 4) | op) for op, ln in cigar) + bytes(packed) + bytes(qual) + aux
  return struct.pack('<i', len(body)) + body


def _bam(records, refs=(('chr20', 1000000), ('chr21', 900000))):
  hdr = b'BAM\1' + struct.pack('<i', 0) + struct.pack('<i', len(refs))
  for name, ln in refs:
    hdr += struct.pack('<i', len(name) + 1) + name.encode() + b'\0' + struct.pack('<i', ln)
  return _bgzf(hdr + b''.join(records))


def _same(a, b):
  assert len(a) == len(b)
  for x, y in zip(a, b):
    assert x == y, (x, y)


def test_hand_built_bam_fields_filters_and_hp(tmp_path):
  recs = [
      _record(0, 100, 'frag1', 60, 0x1 | 0x2 | 0x40, [(0, 5), (1, 2), (0, 3)], 'ACGTNACGTA', range(10, 20), 0, 300, 350),
      _record(0, 120, 'frag1', 50, 0x1 | 0x2 | 0x80 | 0x10, [(4, 2), (0, 6), (2, 3), (0, 2)], 'TTGCAAGGCC', [30] * 10, 0, 100, -350,
              aux=b'NMC\x01' + b'HPC\x02' + b'RGZgrp\0'),
      _record(0, 130, 'dup', 60, 0x400, [(0, 4)], 'ACGT', [40] * 4),                 # duplicate: dropped
      _record(0, 140, 'lowmq', 3, 0, [(0, 4)], 'ACGT', [40] * 4),                    # mapq < 5: dropped
      _record(0, 150, 'farmate', 60, 0x1, [(0, 4)], 'ACGT', [40] * 4, 1, 5000, 0),   # mate on another contig, not proper: dropped
      _record(0, 160, 'matex', 60, 0x1 | 0x8, [(0, 4)], 'ACGT', [40] * 4, 1, 5000, 0),   # mate unmapped: kept
      _record(-1, -1, 'unmapped', 0, 0x4, [], 'ACGT', [40] * 4),                     # unaligned: dropped
      _record(1, 7, 'odd', 60, 0, [(7, 3), (8, 1), (3, 10), (0, 1)], 'ACGTA', [1, 2, 3, 4, 5], aux=b'HPi' + struct.pack('<i', -7)),
      _record(0, 170, 'supp', 60, 0x800, [(0, 4)], 'ACGT', [40] * 4),                # supplementary: dropped
  ]
  path = str(tmp_path / 'tiny.bam')
  open(path, 'wb').write(_bam(recs))
  t = bam.NativeBamTable(path, parse_aux=True)
  assert t.n_records_seen == 9 and t.n_reads == 4 and t.references == ['chr20', 'chr21']
  py = bam.BamReader(path, parse_aux=True)
  _same(t.reads(), py.reads)
  r0, r1, r2, r3 = t.reads()
  assert r0.aligned_sequence == b'ACGTNACGTA' and r0.aligned_quality == bytes(range(10, 20)) and r0.read_number == 0
  assert r0.cigar == [(0, 5), (1, 2), (0, 3)] and r0.fragment_length == 350 and r0.number_reads == 2 and r0.hp_values is None
  assert r1.read_number == 1 and r1.reverse_strand and r1.hp_values == [2] and r1.end() == 120 + 6 + 3 + 2
  assert r2.fragment_name == 'matex'
  assert r3.reference_name == 'chr21' and r3.hp_values == [-7] and int(t.end[3]) == 7 + 3 + 1 + 10 + 1
  np.testing.assert_array_equal(t.end, [r.end() for r in t.reads()])
  # region query == the Python reader's (ReadOverlapsRegion)
  for (c, s, e) in [('chr20', 0, 1000), ('chr20', 108, 121), ('chr20', 131, 132), ('chr21', 0, 8), ('chr21', 22, 23), ('chrX', 0, 9)]:
    _same(t.query(c, s, e), py.query(c, s, e))
  keep_all = bam.ReadRequirements(min_mapping_quality=0, keep_duplicates=True, keep_failed_vendor_quality_checks=True,
                                  keep_secondary_alignments=True, keep_supplementary_alignments=True, keep_unaligned=True,
                                  keep_improperly_placed=True)
  t2 = bam.NativeBamTable(path, keep_all)
  assert t2.n_reads == 9
  _same(t2.reads(), bam.BamReader(path, keep_all).reads)


def test_rejects_garbage(tmp_path):
  from deepvariant_b200 import _lib
  p = str(tmp_path / 'x.bam')
  open(p, 'wb').write(b'not a bam file at all, sorry' * 3)
  with pytest.raises(_lib.DvbError):
    bam.NativeBamTable(p)
  open(p, 'wb').write(_bgzf(b'SAM\1' + b'\0' * 16))
  with pytest.raises(_lib.DvbError):
    bam.NativeBamTable(p)
  with pytest.raises(_lib.DvbError):
    bam.NativeBamTable(str(tmp_path / 'missing.bam'))


# records at the head of each of the reference's test BAMs kept in tests/golden/reads_head.<name> (tools/make_reference_subset_fixtures.py)
HEAD_RECORDS = {'NA12878_S1.chr20.10_10p1mb.bam': 400, 'test_pacbio.chr20_100kbp_at_9mb.bam': 16, 'HG002.hifi.hg37.phased.chr20.1_1000000.bam': 16}


@pytest.mark.parametrize('name,aux', [('NA12878_S1.chr20.10_10p1mb.bam', False), ('test_pacbio.chr20_100kbp_at_9mb.bam', True),
                                     ('HG002.hifi.hg37.phased.chr20.1_1000000.bam', True)])
def test_reference_testdata_identical_to_python_reader(name, aux):
  """The first records of the reference's own test BAMs, byte for byte: the native table and the pure-Python reader agree field by field."""
  path = os.path.join(GOLDEN, 'reads_head.' + name)
  t = bam.NativeBamTable(path, parse_aux=aux)
  py = bam.BamReader(path, parse_aux=aux)
  assert t.n_records_seen == HEAD_RECORDS[name] and t.n_reads == len(py.reads) > 0
  _same(t.reads(), py.reads)
  np.testing.assert_array_equal(t.end, np.array([r.end() for r in py.reads], dtype=np.int32))


def _wgs_generator(ref_reader):
  from deepvariant_b200 import make_examples_native as men, pileup_image as pi
  pic = pi.default_options(pi.ReadRequirements(min_base_quality=10, min_mapping_quality=5))
  pic.channels = list(pi.PILEUP_CHANNELS_WITH_INSERT_SIZE)
  pic.num_channels = 7
  return men.ExamplesGenerator(men.MakeExamplesOptions(pic_options=pic), test_mode=True, ref_reader=ref_reader), pi.to_params(pic)


def _assert_batches_equal(a, b):
  assert (a.n_images, a.n_reads, a.n_pairs, a.ref_stride) == (b.n_images, b.n_reads, b.n_pairs, b.ref_stride)
  for k in a.arrays:
    np.testing.assert_array_equal(a.arrays[k], b.arrays[k], err_msg=k)


def test_table_path_packs_the_same_batch_as_the_read_path_on_the_reference_candidates():
  """The reference's 78 golden candidates over the reads of its NA12878 test BAM in chr20:9,999,000-10,011,000 (quickstart.chr20_10mb.bam,
  a copy re-written with every read kept and the flags rebuilt), partition by partition as make_examples walks them: DvbBatch arrays from
  the table path (row numbers into the native read table) == arrays from Read objects."""
  from deepvariant_b200 import fasta, packing, protos, tfrecord
  cands = [protos.parse_deepvariant_call(r) for r in tfrecord.read_records(os.path.join(GOLDEN, 'golden.calling_candidates.tfrecord.gz'))]
  path = os.path.join(GOLDEN, 'quickstart.chr20_10mb.bam')
  req = bam.ReadRequirements(min_mapping_quality=5)
  reader, table = bam.BamReader(path, req), bam.NativeBamTable(path, req)
  gen, params = _wgs_generator(fasta.IndexedFastaReader(os.path.join(GOLDEN, 'quickstart.chr20_10mb.fa.gz')))
  region_start, part = 9_999_999, 1000
  by_part = {}
  for c in cands:
    by_part.setdefault(region_start + (c.variant.start - region_start) // part * part, []).append(c)
  n_images = 0
  for p0, cs in sorted(by_part.items()):
    region = (cs[0].variant.reference_name, p0, min(p0 + part, 10_010_000))
    plans = gen.plan_region(cs, reader.query(*region), {})
    want = packing.pack_images([p.spec for p in plans], params)
    plans_t, specs = gen.plan_region_from_table(cs, table, {}, region)
    got = packing.pack_images_from_table(specs, table, params)
    assert [(p.variant.start, p.alt_combination, p.variant_type) for p in plans] == \
        [(p.variant.start, p.alt_combination, p.variant_type) for p in plans_t]
    _assert_batches_equal(got, want)
    plans_n, native = gen.pack_region_native(cs, table, region)   # C++ region packer
    assert [(p.variant.start, p.alt_combination) for p in plans_n] == [(p.variant.start, p.alt_combination) for p in plans]
    _assert_batches_equal(native, want)
    n_images += got.n_images
  assert n_images == 84   # the reference's golden.calling_examples has 84 examples for these candidates


def test_table_path_on_a_hand_built_bam(tmp_path):
  """Portable version of the test above: synthetic reads + candidates with allele support, multi-allelic included."""
  from deepvariant_b200 import packing, protos
  rng = np.random.default_rng(5)
  recs = []
  for i in range(60):
    pos = 400 + int(rng.integers(0, 300))
    seq = ''.join(rng.choice(list('ACGT'), 50))
    paired = i % 3 != 0
    flag = (0x1 | 0x2 | (0x40 if i % 2 else 0x80)) if paired else 0
    flag |= 0x10 if i % 5 == 0 else 0
    cigar = [(0, 50)] if i % 7 else [(0, 20), (1, 5), (0, 25)]
    recs.append((pos, _record(0, pos, f'r{i // 2}' if paired else f's{i}', 20 + i % 40, flag, cigar, seq, rng.integers(5, 41, 50).tolist(),
                              0 if paired else -1, pos + 100 if paired else -1, 150 if i % 2 else -150)))
  recs.sort(key=lambda t: t[0])
  path = str(tmp_path / 'syn.bam')
  open(path, 'wb').write(_bam([r for _, r in recs]))
  reader, table = bam.BamReader(path), bam.NativeBamTable(path)

  class Ref:
    def n_bases(self, contig): return 1000000
    def is_valid_interval(self, contig, s, e): return 0 <= s < e <= 1000000
    def query(self, contig, s, e): return ('ACGT' * 250001)[s:e]
  gen, params = _wgs_generator(Ref())
  keys = [r.key() for r in reader.reads]
  cands = []
  for start, alts in [(450, ['T']), (520, ['G', 'GA']), (610, ['C']), (699, ['T', 'A'])]:
    v = protos.Variant(reference_name='chr20', start=start, end=start + 1, reference_bases='A', alternate_bases=list(alts))
    sup = {a: [keys[(start + 7 * j + 3 * k) % len(keys)] for j in range(6)] for k, a in enumerate(alts)}
    cands.append(protos.DeepVariantCall(variant=v, allele_support=sup))
  region = ('chr20', 400, 800)
  plans = gen.plan_region(cands, reader.query(*region), {})
  plans_t, specs = gen.plan_region_from_table(cands, table, {}, region)
  assert len(plans) == len(plans_t) == 1 + 3 + 1 + 3
  want = packing.pack_images([p.spec for p in plans], params)
  _assert_batches_equal(packing.pack_images_from_table(specs, table, params), want)
  plans_n, native = gen.pack_region_native(cands, table, region)
  assert len(plans_n) == len(plans)
  _assert_batches_equal(native, want)
  # allele-support sorting on (pair_allele_group filled), a region that cuts reads off, a candidate on another contig
  gen.options.pic_options.sort_by_alt_allele_support = True
  other = protos.DeepVariantCall(variant=protos.Variant(reference_name='chrX', start=500, end=501, reference_bases='A', alternate_bases=['C']),
                                 allele_support={'C': keys[:3]})
  for region in (('chr20', 400, 800), ('chr20', 500, 620), ('chr20', 0, 10)):
    cs = cands + [other]
    plans = gen.plan_region(cs, reader.query(*region), {})
    want = packing.pack_images([p.spec for p in plans], params)
    _, specs = gen.plan_region_from_table(cs, table, {}, region)
    _assert_batches_equal(packing.pack_images_from_table(specs, table, params), want)
    _, native = gen.pack_region_native(cs, table, region)
    _assert_batches_equal(native, want)
  assert want.arrays['pair_allele_group'].max() >= 0
  # no candidates at all
  _, empty = gen.pack_region_native([], table, ('chr20', 400, 800))
  assert (empty.n_images, empty.n_reads, empty.n_pairs) == (0, 0, 0)


@pytest.mark.parametrize('seed,coordinate_sorted', [(1, True), (2, False), (3, True), (4, False)])
def test_region_packer_equals_numpy_packer_on_random_bams(tmp_path, seed, coordinate_sorted):
  """C++ region packer == numpy table packer on random files: two contigs, unsorted files (linear scan instead of the
  binary search), the same QNAME aligned twice, reads with very different spans, support keys that name no read or are
  not of the "name/0|1" form, regions that clip the read set, sort_by_alt_allele_support on and off."""
  from deepvariant_b200 import packing, protos
  rng = np.random.default_rng(seed)
  recs = []
  for i in range(300):
    ref_id = int(rng.integers(0, 2))
    pos = 1000 + int(rng.integers(0, 1500))
    ln = int(rng.choice([30, 80, 400]))
    seq = ''.join(rng.choice(list('ACGT'), ln))
    paired = i % 4 != 0
    flag = (0x1 | 0x2 | (0x40 if i % 2 else 0x80)) if paired else 0
    name = f'q{int(rng.integers(0, 120))}'            # few names: several alignments share a key
    cigar = [(0, ln)] if i % 5 else [(0, 10), (2, 7), (0, ln - 10)]
    recs.append(((ref_id, pos), _record(ref_id, pos, name, 10 + i % 50, flag, cigar, seq, rng.integers(5, 41, ln).tolist(),
                                        ref_id if paired else -1, pos + 50 if paired else -1, 200)))
  if coordinate_sorted:
    recs.sort(key=lambda t: t[0])
  path = str(tmp_path / f'rand{seed}.bam')
  open(path, 'wb').write(_bam([r for _, r in recs]))
  table = bam.NativeBamTable(path)
  keys = [r.key() for r in table.reads()]

  class Ref:
    def n_bases(self, contig): return 1000000
    def is_valid_interval(self, contig, s, e): return 0 <= s < e <= 1000000
    def query(self, contig, s, e): return ('ACGT' * 250001)[s:e]
  gen, params = _wgs_generator(Ref())
  cands = []
  for k in range(12):
    contig = 'chr20' if k % 3 else 'chr21'
    start = 1000 + int(rng.integers(0, 1600))
    alts = ['T', 'TA', 'G'][:1 + k % 3]
    sup = {a: [keys[int(j)] for j in rng.integers(0, len(keys), 8)] + ['nobody/0', 'noslash', keys[0] + '1', keys[1][:-1] + '2', '']
           for a in alts}
    v = protos.Variant(reference_name=contig, start=start, end=start + 1 + k % 2, reference_bases='A' * (1 + k % 2), alternate_bases=alts)
    cands.append(protos.DeepVariantCall(variant=v, allele_support=sup))
  for sort_by_support in (False, True):
    gen.options.pic_options.sort_by_alt_allele_support = sort_by_support
    for region in (('chr20', 900, 3000), ('chr21', 1500, 1700), ('chr20', 2400, 2401), ('chr21', 0, 5)):
      plans_t, specs = gen.plan_region_from_table(cands, table, {}, region)
      want = packing.pack_images_from_table(specs, table, params)
      plans_n, got = gen.pack_region_native(cands, table, region)
      assert [(p.variant.start, p.alt_combination) for p in plans_n] == [(p.variant.start, p.alt_combination) for p in plans_t]
      _assert_batches_equal(got, want)
  assert want.n_images > 12


def test_region_packer_argument_errors(tmp_path):
  from deepvariant_b200 import _lib, packing, pileup_image as pi
  path = str(tmp_path / 'one.bam')
  open(path, 'wb').write(_bam([_record(0, 100, 'a', 60, 0, [(0, 4)], 'ACGT', [40] * 4)]))
  table = bam.NativeBamTable(path)
  params = pi.to_params(pi.default_options())
  im = packing.RegionImage(0, 100, 101, 100 - 110, b'A' * (params.width - 1), b'a/0', np.array([3], np.int64), np.array([1], np.uint8))
  with pytest.raises(ValueError):
    packing.pack_region_native(table, [im], 0, 0, 1000, 5, params)
  im.ref_bases = b'A' * params.width
  b = packing.pack_region_native(table, [im], 0, 0, 1000, 5, params)
  assert (b.n_images, b.n_reads, b.n_pairs) == (1, 1, 1) and b.arrays['pair_support'][0] == 1
  table.close()
  with pytest.raises(ValueError):
    packing.pack_region_native(table, [im], 0, 0, 1000, 5, params)


def _cli_from_bam_file_matches_oracle(tmp_path):
  """The make_examples stage CLI end to end on files: BAM (native decode -> table path) + indexed FASTA + candidates TFRecord
  -> examples TFRecord; every image/encoded equals the CPU oracle's encoding of the same candidate planned from the
  pure-Python reader's Read objects."""
  import oracle_lib
  from deepvariant_b200 import cli, packing, protos, tfrecord
  from deepvariant_b200 import make_examples_native as men
  rng = np.random.default_rng(11)
  contig_len = 5000
  genome = ''.join(rng.choice(list('ACGT'), contig_len))
  fa = tmp_path / 'ref.fa'
  fa.write_text('>chr20\n' + '\n'.join(genome[i:i + 60] for i in range(0, contig_len, 60)) + '\n')
  (tmp_path / 'ref.fa.fai').write_text(f'chr20\t{contig_len}\t7\t60\t61\n')
  recs = []
  for i in range(400):
    pos = 1000 + int(rng.integers(0, 2000))
    seq = list(genome[pos:pos + 100])
    for j in rng.integers(0, 100, 2):
      seq[j] = 'ACGT'[int(rng.integers(0, 4))]
    flag = 0x1 | 0x2 | (0x40 if i % 2 else 0x80) | (0x10 if i % 3 == 0 else 0)
    recs.append((pos, _record(0, pos, f'q{i // 2}', int(rng.integers(0, 61)), flag, [(0, 100)], ''.join(seq), rng.integers(2, 41, 100).tolist(),
                              0, pos + 150, 250 if i % 2 else -250)))
  recs.sort(key=lambda t: t[0])
  bam_path = str(tmp_path / 'reads.bam')
  open(bam_path, 'wb').write(_bam([r for _, r in recs], refs=(('chr20', contig_len),)))
  reader = bam.BamReader(bam_path)
  cands = []
  for start in (1100, 1500, 1999, 2000, 2700, 2950):
    ov = [r.key() for r in reader.query('chr20', start, start + 1)]
    alts = ['T'] if start % 200 else ['T', 'TG']
    sup = {a: ov[k::3][:8] for k, a in enumerate(alts)}
    v = protos.Variant(reference_name='chr20', start=start, end=start + 1, reference_bases=genome[start], alternate_bases=alts)
    cands.append(protos.DeepVariantCall(variant=v, allele_support=sup))
  cpath = str(tmp_path / 'cands.tfrecord.gz')
  w = tfrecord.Writer(cpath)
  for c in cands:
    w.write(protos.serialize_deepvariant_call(c))
  w.close()
  ex = str(tmp_path / 'make_examples.tfrecord@1.gz')
  assert cli.make_examples(['--mode', 'calling', '--ref', str(fa), '--reads', bam_path, '--candidates_in', cpath, '--examples', ex,
                            '--channel_list', 'BASE_CHANNELS,insert_size', '--regions', 'chr20:1001-3000']) == 0
  got = [protos.parse_tf_example(r) for r in tfrecord.read_records(str(tmp_path / 'make_examples.tfrecord-00000-of-00001.gz'))]
  # expected: Read-object planner + CPU oracle, partition by partition (1000-bp partitions from the region start)
  from deepvariant_b200 import fasta
  gen, params = _wgs_generator(fasta.IndexedFastaReader(str(fa)))
  want_imgs, want_keys = [], []
  for p0 in (1000, 2000):
    cs = [c for c in cands if p0 <= c.variant.start < p0 + 1000]
    plans = gen.plan_region(cs, reader.query('chr20', p0, p0 + 1000), {})
    imgs = oracle_lib.encode_batch(params, packing.pack_images([p.spec for p in plans], params))
    want_imgs += list(imgs)
    want_keys += [(p.variant.start, men.encode_alt_alleles(p.variant, p.alt_combination)[0]) for p in plans]
  assert len(got) == len(want_imgs), (len(got), len(want_imgs))
  assert len(got) == 5 * 1 + 1 * 3, len(got)   # five bi-allelic candidates + one with two alts (3 combinations)
  for e, img, (start, alt_enc) in zip(got, want_imgs, want_keys):
    assert protos.parse_variant(e['variant/encoded'][1][0]).start == start
    assert e['alt_allele_indices/encoded'][1][0] == alt_enc
    assert e['image/shape'][1] == [100, 221, 7]
    np.testing.assert_array_equal(np.frombuffer(e['image/encoded'][1][0], np.uint8).reshape(100, 221, 7), img)


@pytest.mark.gpu
def test_make_examples_cli_from_bam_file_matches_oracle(tmp_path):
  _cli_from_bam_file_matches_oracle(tmp_path)


def test_make_examples_cli_from_bam_file_cpu_plumbing(tmp_path, monkeypatch):
  """The same flow with the encoder replaced by the CPU oracle: everything around the CUDA call (flags, --candidates_in,
  partitions, native table path, serialisation) runs on the CPU suite too."""
  import oracle_lib
  from deepvariant_b200 import make_examples_native as men, pileup_image as pi

  class OracleEncoder:
    def __init__(self, params):
      self.params = params
      self.shape = (params.height, params.width, params.num_channels + params.num_alt_channels)

    def encode_host(self, batch):
      return oracle_lib.encode_batch(self.params, batch)

  monkeypatch.setattr(men.ExamplesGenerator, '_gpu', lambda self: OracleEncoder(pi.to_params(self.options.pic_options, height=self.pileup_image_height)))
  _cli_from_bam_file_matches_oracle(tmp_path)


def _assert_same_rows(sub, full, keep):
  import numpy as np
  assert sub.n_reads == int(keep.sum())
  for name in ('ref_id', 'pos', 'end', 'mapq', 'flag', 'fragment_length', 'read_number'):
    np.testing.assert_array_equal(getattr(sub, name), getattr(full, name)[keep], err_msg=name)
  idx = np.nonzero(keep)[0]
  for k in (0, len(idx) // 2, len(idx) - 1):
    if len(idx):
      assert sub.read(k).key() == full.read(int(idx[k])).key() and sub.read(k).aligned_sequence == full.read(int(idx[k])).aligned_sequence


def test_region_restricted_open_equals_the_filtered_full_table(tmp_path):
  """dvb_bam_open_regions: (a) an un-indexed synthetic file (scan + filter, several regions on two contigs, a contig the file does not
  know), (b) the reference's indexed chr20 test BAM through its .bai linear index (one region: decoding starts at the indexed block and
  stops behind the region) - both against the full table filtered with ReadOverlapsRegion; sorted-table region queries (two binary
  searches) against the scan."""
  import numpy as np
  from deepvariant_b200 import bam
  rng = np.random.default_rng(3)
  recs = []
  for ref, n in ((0, 900), (1, 400)):
    for pos in np.sort(rng.integers(0, 20000, n)).tolist():
      L = int(rng.integers(30, 151))
      recs.append(_record(ref, pos, f'r{len(recs)}', 60, 0, [(0, L)], ''.join(rng.choice(list('ACGT'), L)), rng.integers(5, 41, L).tolist()))
  path = str(tmp_path / 'two.bam')
  open(path, 'wb').write(_bam(recs, refs=(('chr1', 30000), ('chr2', 30000))))
  reqs = bam.ReadRequirements(min_mapping_quality=5)
  full = bam.NativeBamTable(path, reqs)
  regions = [('chr1', 1000, 1500), ('chr2', 300, 320), ('chr1', 15000, 15010), ('chrUn', 0, 100)]
  keep = np.zeros(full.n_reads, dtype=bool)
  for c, s, e in regions[:3]:
    rid = full.references.index(c)
    keep |= (full.ref_id == rid) & (full.pos < e) & (full.end > s)
  _assert_same_rows(bam.NativeBamTable(path, reqs, regions=regions), full, keep)
  assert bam.NativeBamTable(path, reqs, regions=[('chrUn', 0, 100)]).n_reads == 0
  for c, s, e in (('chr1', 0, 1), ('chr1', 1000, 1500), ('chr2', 19990, 30000), ('chr2', 5000, 5001), ('chr1', 29999, 30000)):
    rid = full.references.index(c)
    np.testing.assert_array_equal(full.query_indices(c, s, e), np.nonzero((full.ref_id == rid) & (full.pos < e) & (full.end > s))[0])
  # real reads: the records of the reference's NA12878 test BAM that start before chr20:10,011,000, with their .bai
  real = os.path.join(GOLDEN, 'NA12878_S1.chr20.10_10p1mb.window.bam')
  full = bam.NativeBamTable(real, reqs)
  for s, e in ((10_000_000, 10_010_000), (10_005_123, 10_005_124), (10_010_700, 10_011_000), (9_000_000, 9_500_000)):
    rid = full.references.index('chr20')
    keep = (full.ref_id == rid) & (full.pos < e) & (full.end > s)
    sub = bam.NativeBamTable(real, reqs, regions=[('chr20', s, e)])
    _assert_same_rows(sub, full, keep)
    if keep.any() and s > 10_010_624:      # past the first 16-kb window of the linear index the file holds reads of
      assert sub.n_records_seen < full.n_records_seen // 2, 'the index was not used: the whole file was parsed'


def test_malformed_bgzf_headers_are_rejected_not_overrun(tmp_path):
  """BSIZE smaller than header + trailer (the subtraction would wrap), an extra field running past the block, a missing BC subfield."""
  from deepvariant_b200 import _lib, bam
  good = _bam([_record(0, 5, 'a', 60, 0, [(0, 10)], 'ACGTACGTAC', [30] * 10)])
  for name, blob in (
      ('tiny_bsize', good[:16] + (5).to_bytes(2, 'little') + good[18:]),
      ('xlen_overrun', good[:10] + (60000).to_bytes(2, 'little') + good[12:]),
      ('no_bc', good[:12] + b'XY' + good[14:]),
  ):
    p = tmp_path / f'{name}.bam'
    p.write_bytes(blob)
    with pytest.raises(_lib.DvbError):
      bam.NativeBamTable(str(p))


@pytest.mark.parametrize('seed', [1, 2])
def test_derived_table_equals_the_scratch_bam_table(tmp_path, seed):
  """dvb_bam_derive (realigned / normalised reads as a table of their own) against the path through a temporary BAM: the same reads in the
  same order, new alignments applied, everything else of the records copied; a region query, the native packer's view and the errors."""
  import copy
  rng = np.random.default_rng(seed)
  recs = []
  for i in range(200):
    pos = 1000 + int(rng.integers(0, 1500))
    ln = int(rng.choice([30, 80, 150]))
    paired = i % 4 != 0
    flag = (0x1 | 0x2 | (0x40 if i % 2 else 0x80) | (0x20 if i % 3 == 0 else 0)) if paired else (0x10 if i % 2 else 0)
    cigar = [(0, ln)] if i % 5 else [(4, 3), (0, 7), (2, 7), (0, ln - 10)]
    aux = b'HPi' + (1 + i % 2).to_bytes(4, 'little') if i % 3 == 0 else b''
    recs.append((pos, _record(0, pos, f'q{i // 2}', 10 + i % 50, flag, cigar, ''.join(rng.choice(list('ACGTN'), ln)), rng.integers(5, 41, ln).tolist(),
                              0 if paired else -1, pos + 50 if paired else -1, 200, aux)))
  recs.sort(key=lambda t: t[0])
  path = str(tmp_path / f'derive{seed}.bam')
  open(path, 'wb').write(_bam([r for _, r in recs]))
  table = bam.NativeBamTable(path, bam.ReadRequirements(min_mapping_quality=12), parse_aux=True)
  rows = rng.permutation(table.query_indices('chr20', 1200, 2300))          # the realigner reorders reads
  reads = [copy.copy(table.read(int(i))) for i in rows]
  changed = 0
  for k, r in enumerate(reads):
    if k % 3 == 0 and len(r.aligned_sequence) > 20:
      n = len(r.aligned_sequence)
      r.position += int(rng.integers(-5, 20))
      r.cigar = [(4, 2), (0, 8), (1, 3), (0, n - 16), (2, 4), (0, 3)]
      changed += 1
  assert changed > 10
  refs = list(zip(table.references, table.reference_lengths))
  derived = bam.scratch_table(reads, refs, bam.ReadRequirements(min_mapping_quality=12), parse_aux=True)     # every read carries its source row
  for r in reads:
    del r._table, r._row
  scratch = bam.scratch_table(reads, refs, bam.ReadRequirements(min_mapping_quality=12), parse_aux=True)     # ... and now none does: temporary BAM
  assert derived.n_reads == scratch.n_reads == len(reads)
  assert derived.reads() == scratch.reads() == reads
  for name in ('ref_id', 'pos', 'end', 'mapq', 'fragment_length', 'hp', 'read_number', 'number_reads', 'seq_begin', 'cigar_begin', 'name_begin',
               'bases', 'quals', 'cigar'):
    np.testing.assert_array_equal(getattr(derived, name), getattr(scratch, name), err_msg=name)
  assert derived.names == scratch.names and derived.references == scratch.references and derived.reference_lengths == scratch.reference_lengths
  np.testing.assert_array_equal(derived.query_indices('chr20', 1500, 1600), scratch.query_indices('chr20', 1500, 1600))
  same = bam.NativeBamTable.derived(table, rows)                                     # no new alignments: a plain sub-table
  assert same.reads() == [table.read(int(i)) for i in rows]
  assert bam.NativeBamTable.derived(table, []).n_reads == 0
  with pytest.raises(_lib.DvbError, match='out of range'):
    bam.NativeBamTable.derived(table, [table.n_reads])
  with pytest.raises(_lib.DvbError, match='consumes'):
    bam.NativeBamTable.derived(table, rows[:1], [(5, [(0, 7)])])
  with pytest.raises(_lib.DvbError, match='CIGAR operation'):
    bam.NativeBamTable.derived(table, rows[:1], [(5, [(9, len(reads[0].aligned_sequence))])])
  with pytest.raises(ValueError):
    bam.NativeBamTable.derived(table, rows[:2], [None])
