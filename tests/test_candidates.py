"""Candidate generation (csrc/dvb_candidates.cu + deepvariant_b200/candidates.py; SURVEY 8(f) next row #2).

  * known-answer tests transcribed as data from deepvariant/allelecounter_test.cc:329-1065 and
    deepvariant/variant_calling_test.cc:328-760, run against the C++ product (reads go through a hand-built BAM and the
    native table) and against the Python restatement oracle/candidates_oracle.py;
  * product == oracle on random reads (indels, clips, N bases, low qualities, repeated read keys, track_ref_reads);
  * the reference's golden files: a portable fixture cut from golden.calling_candidates (tools/check_candidates_golden.py)
    and the variants of golden.pacbio_examples in a 5-kb window (tools/make_reference_subset_fixtures.py).
CPU-only: host code of libdvb.so."""
import json
import os
import random
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import candidates_oracle as oc  # noqa: E402
import test_bam_native as tb  # noqa: E402
from deepvariant_b200 import bam, candidates as cand, protos  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
# third_party/nucleus/testdata/test.fasta, the contigs allelecounter_test.cc uses
CHR1 = b'ACCACCATCCTCCGTGAAATCAATATCCCGCACAAGAGTGCTACTCTCCTAAATCCCTTCTCGTCCCCATGGATGA'
CHR2 = b'CGCTNCGGGCCCATAACACTTGGGGGTAGCTAAAGTGAACTGTATCC'
R, S, I, D, C = oc.REFERENCE, oc.SUBSTITUTION, oc.INSERTION, oc.DELETION, oc.SOFT_CLIP


class FakeRef:
  def __init__(self, contigs):
    self.contigs = dict(contigs)
    self.contig_order = [c for c, _ in contigs]

  def _contig(self, name):
    return self.contigs[name]

  def n_bases(self, name):
    return len(self.contigs[name])


def _read(name, pos, seq, cigar, quals=None, mapq=90, number=0, reverse=False):
  cig = protos.parse_cigar_string(cigar)
  return protos.Read(fragment_name=name, read_number=number, reference_name='', position=pos, reverse_strand=reverse,
                     mapping_quality=mapq, cigar=cig, aligned_sequence=seq.encode(),
                     aligned_quality=bytes(quals if quals is not None else [30] * len(seq)))


def _table(tmp_path, reads, contigs, ref_id=0):
  recs = []
  for r in reads:
    flag = (0x10 if r.reverse_strand else 0) | ((0x1 | (0x80 if r.read_number else 0x40)) if r.read_number or getattr(r, '_paired', False) else 0)
    recs.append(tb._record(ref_id, r.position, r.fragment_name, r.mapping_quality, flag, r.cigar, r.aligned_sequence.decode(),
                           r.aligned_quality))
  path = str(tmp_path / f'reads{random.getrandbits(32)}.bam')
  with open(path, 'wb') as f:
    f.write(tb._bam(recs, refs=tuple((c, len(b)) for c, b in contigs)))
  req = bam.ReadRequirements(min_mapping_quality=0)
  req.keep_unaligned = True
  return bam.NativeBamTable(path, req)


def _summed(site, ref_base):
  """SumAlleleCounts incl. the synthetic reference allele -> sorted [(bases, type, count)]."""
  m = {}
  for bases, typ, low, *_ in site['alleles']:
    if not low:
      m[(bases, typ)] = m.get((bases, typ), 0) + 1
  if site['ref'] > 0:
    m[(ref_base, R)] = site['ref']
  return sorted((b, t, n) for (b, t), n in m.items())


def _oracle_summed(ac):
  m = {(a['bases'], a['type']): a['count'] for a in oc.sum_allele_counts(ac)}
  if ac.ref_supporting_read_count > 0:
    m[(ac.ref_base, R)] = ac.ref_supporting_read_count
  return sorted((b, t, n) for (b, t), n in m.items())


def _check_counts(tmp_path, reads, expected, contig=('chr1', CHR1), start=10, end=15, min_bq=21, min_mapq=5):
  """AddAndCheckReads (allelecounter_test.cc:149-193) on both implementations."""
  ref = FakeRef([('chr1', CHR1), ('chr2', CHR2)])
  name, bases = contig
  opts = cand.CandidateOptions(min_base_quality=min_bq, min_mapping_quality=min_mapq)
  table = _table(tmp_path, reads, [('chr1', CHR1), ('chr2', CHR2)], ref_id=0 if name == 'chr1' else 1)
  got = cand.debug_allele_counts(table, ref, name, start, end, np.arange(table.n_reads), opts)
  want = [sorted(e) for e in expected]
  assert [_summed(s, bases[start + i:start + i + 1].decode()) for i, s in enumerate(got)] == want
  counter = oc.AlleleCounter(bases, start, end, oc.Options(min_base_quality=min_bq, min_mapping_quality=min_mapq))
  for r in reads:
    counter.add(r)
  assert [_oracle_summed(ac) for ac in counter.counts] == want
  table.close()


REF5 = [[('T', R, 1)], [('C', R, 1)], [('C', R, 1)], [('G', R, 1)], [('T', R, 1)]]


def _ref5(**replace):
  out = [list(x) for x in REF5]
  for k, v in replace.items():
    out[int(k[1:])] = v
  return out


ALLELE_COUNTER_KATS = [
    # (name, [(pos, seq, cigar)], expected per position)                      allelecounter_test.cc
    ('simple_M', [(10, 'TCCGT', '5M')], REF5),                                                      # :329
    ('simple_X', [(10, 'TCCGT', '5X')], REF5),
    ('simple_EQ', [(10, 'TCCGT', '5=')], REF5),
    ('beyond_interval', [(8, 'AATCCGTAA', '9M')], REF5),                                            # :342
    ('substitution', [(10, 'TCAGT', '5M')], _ref5(p2=[('A', S, 1)])),                               # :520
    ('insertion1', [(10, 'TCAAACGT', '2M3I3M')], _ref5(p1=[('CAAA', I, 1)])),                       # :534
    ('insertion2', [(10, 'TAAACCGT', '1M3I4M')], _ref5(p0=[('TAAA', I, 1)])),                       # :545
    ('insertion3', [(10, 'TCCGTAAA', '5M3I')], _ref5(p4=[('TAAA', I, 1)])),                         # :556
    ('start_insertion_dropped', [(10, 'AAATCCGT', '3I5M')], REF5),                                  # :583
    ('start_insertion_kept', [(11, 'AAACCGT', '3I4M')], _ref5(p0=[('TAAA', I, 1)])),                # :595
    ('deletion1', [(10, 'TCGT', '2M1D2M')], _ref5(p1=[('CC', D, 1)], p2=[])),                       # :608
    ('starting_deletion_dropped', [(10, 'CCGT', '1D4M')], _ref5(p0=[])),                            # :674
    ('starting_deletion_kept', [(11, 'CGT', '1D3M')], _ref5(p0=[('TC', D, 1)], p1=[])),
    ('deletion_to_end', [(10, 'TCCG', '4M1D')], _ref5(p3=[('GT', D, 1)], p4=[])),                   # :698
    ('deletion_off_interval', [(10, 'TCCG', '4M3D')], _ref5(p3=[('GTGA', D, 1)], p4=[])),           # :710
    ('multiple_reads', [(10, 'TCCGT', '5M'), (10, 'TCGT', '2M1D2M'), (12, 'CGT', '3M'), (10, 'TCCAGT', '3M1I2M'), (12, 'CG', '2M')],
     [[('T', R, 3)], [('C', R, 2), ('CC', D, 1)], [('C', R, 3), ('CA', I, 1)], [('G', R, 5)], [('T', R, 4)]]),   # :723
    ('softclip1', [(12, 'AACGT', '2S3M')], _ref5(p0=[], p1=[('CAA', C, 1)])),                       # :745
    ('softclip2', [(11, 'ACCGT', '1S4M')], _ref5(p0=[('TA', C, 1)])),                               # :756
    ('softclip3', [(10, 'AATCCGT', '2S5M')], REF5),                                                 # :767
    ('softclip4', [(10, 'TCCGTAA', '5M2S')], _ref5(p4=[('TAA', C, 1)])),                            # :779
    ('snp_indel', [(10, 'TAAAACGT', '2M3I3M')], _ref5(p1=[('AAAA', I, 1)])),                        # :958
    ('noncanonical_read_base', [(10, 'TCNGT', '5M')], _ref5(p2=[])),                                # :991
    ('noncanonical_prev_base', [(10, 'TNGT', '2M1D2M')], _ref5(p1=[], p2=[])),
    ('noncanonical_prev_base_ins', [(10, 'TCNAGT', '3M1I2M')], _ref5(p2=[])),
    ('noncanonical_inserted_base', [(10, 'TCCNGT', '3M1I2M')], REF5),
]


@pytest.mark.parametrize('name,reads,expected', ALLELE_COUNTER_KATS, ids=[k[0] for k in ALLELE_COUNTER_KATS])
def test_allele_counter_kats(tmp_path, name, reads, expected):
  _check_counts(tmp_path, [_read(f'read_{i}', p, s, c) for i, (p, s, c) in enumerate(reads)], expected)


def test_allele_counter_add_read_all_subranges(tmp_path):
  """TestAddRead (allelecounter_test.cc:353-375)."""
  for start in range(5):
    for end in range(5, start, -1):
      expected = [[(chr(CHR1[10 + i]), R, 1)] if start <= i < end else [] for i in range(5)]
      _check_counts(tmp_path, [_read('r', 10 + start, CHR1[10 + start:10 + end].decode(), f'{end - start}M')], expected)


def test_allele_counter_insertion_sizes_and_deletion_sizes(tmp_path):
  for size in range(1, 10):     # TestDiffInsertionSizes :567
    _check_counts(tmp_path, [_read('r', 10, 'TC' + 'A' * size + 'CGT', f'2M{size}I3M')], _ref5(p1=[('C' + 'A' * size, I, 1)]))


def test_allele_counter_contig_edges(tmp_path):
  """TestInsertionAtChrStart / TestAtChrEnd1 / TestDeletionAtChrStart (:790-851)."""
  for op in ('2S', '2I'):
    _check_counts(tmp_path, [_read('r', 0, 'AAAC', op + '2M')], [[('A', R, 1)], [('C', R, 1)]], start=0, end=2)
  n = len(CHR1)
  for op, typ in (('2S', C), ('2I', I)):
    _check_counts(tmp_path, [_read('r', n - 2, 'GAAA', '2M' + op)], [[('G', R, 1)], [('AAA', typ, 1)]], start=n - 2, end=n)
  _check_counts(tmp_path, [_read('r', n - 2, 'GA', '2M2D')], [[('G', R, 1)], [('A', R, 1)]], start=n - 2, end=n)
  _check_counts(tmp_path, [_read('r', n - 2, 'GAAAAAAA', '8M')], [[('G', R, 1)], [('A', R, 1)]], start=n - 2, end=n)
  _check_counts(tmp_path, [_read('r', 0, 'CA', '2D2M')], [[], [], [('C', R, 1)], [('A', R, 1)]], start=0, end=4)


def test_allele_counter_quality_filters(tmp_path):
  """TestLowMapqReadsAreIgnored, TestMinBaseQualSNP, TestMinBaseQualInsertion, TestMinBaseQualIndelBadInitialBase (:853-956)."""
  _check_counts(tmp_path, [_read('r', 0, 'ACGT', '4M', mapq=0)], [[], [], [], []], start=0, end=4, min_mapq=10)
  for bad in range(5):
    q = [30] * 5
    q[bad] = 20
    _check_counts(tmp_path, [_read('r', 10, 'TCCGT', '5M', q)], _ref5(**{f'p{bad}': []}))
  for bad in (1, 2, 3):
    q = [22] * 5
    q[bad] = 18
    _check_counts(tmp_path, [_read('r', 10, 'TAAAC', '1M3I1M', q)], [[], [('C', R, 1)], [], [], []])
  q = [22] * 8
  q[3] = 17
  _check_counts(tmp_path, [_read('r', 10, 'TCAAACGT', '2M3I3M', q)], _ref5(p1=[]))
  q[1] = 20
  _check_counts(tmp_path, [_read('r', 10, 'TCAAACGT', '2M3I3M', q)], _ref5(p1=[]))
  q[3] = 22
  _check_counts(tmp_path, [_read('r', 10, 'TCAAACGT', '2M3I3M', q)], _ref5(p1=[('CAAA', I, 1)]))


def test_allele_counter_paired_reads_and_reference_n(tmp_path):
  """TestPairedReads (:971) - same fragment, read numbers 0 / 1 are different keys; TestCanonicalBasesReference (:1033)."""
  r1, r2 = _read('fragment', 10, 'TCCAT', '5M', number=0), _read('fragment', 10, 'TCAAT', '5M', number=1)
  r1._paired = True
  _check_counts(tmp_path, [r1, r2], [[('T', R, 2)], [('C', R, 2)], [('C', R, 1), ('A', S, 1)], [('A', S, 2)], [('T', R, 2)]])
  _check_counts(tmp_path, [_read('r', 2, 'CTACG', '5M')], [[('C', R, 1)], [('T', R, 1)], [('A', S, 1)], [('C', R, 1)], [('G', R, 1)]],
                contig=('chr2', CHR2), start=2, end=7)
  _check_counts(tmp_path, [_read('r', 2, 'CTCG', '2M1D2M')], [[('C', R, 1)], [('T', R, 1)], [], [('C', R, 1)], [('G', R, 1)]],
                contig=('chr2', CHR2), start=2, end=7)


# ---- the caller: variant_calling_test.cc:617-760 (alleles at one site -> Variant with AD) ---------------------------------
SITE_REF = b'GGGGGGGGGGATGCATGCATGC' + b'G' * 30     # position 10 = 'A', followed by TGC...


def _reads_for(alleles):
  """One read per supporting observation of (bases, type) at position 10 of SITE_REF."""
  reads = []
  for bases, typ, count in alleles:
    for _ in range(count):
      n = len(reads)
      if typ == R:
        reads.append(_read(f'r{n}', 10, 'AT', '2M'))
      elif typ == S:
        reads.append(_read(f'r{n}', 10, bases + 'T', '2M'))
      elif typ == I:
        reads.append(_read(f'r{n}', 10, bases + 'T', f'1M{len(bases) - 1}I1M'))
      elif typ == D:
        k = len(bases) - 1
        reads.append(_read(f'r{n}', 10, 'A' + SITE_REF[11 + k:12 + k].decode(), f'1M{k}D1M'))
      elif typ == C:
        reads.append(_read(f'r{n}', 9, 'GA' + bases[1:], f'2M{len(bases) - 1}S'))
  return reads


CALLER_KATS = [
    # (name, alleles, min_count, expected (ref, alts, AD) or None)
    ('no_variant', [('A', R, 10)], 3, None),                                                         # :328
    ('no_variant_from_softclips', [('ACCCCC', C, 10)], 3, None),                                     # :337
    ('snp', [('C', S, 10), ('A', R, 10)], 3, ('A', ['C'], [10, 10])),                                # :345
    ('multi_allelic_snp', [('C', S, 10), ('G', S, 10)], 10, ('A', ['C', 'G'], [0, 10, 10])),         # :617
    ('deletion', [('ATGC', D, 10)], 10, ('ATGC', ['A'], [0, 10])),                                   # :630
    ('insertion', [('ACCC', I, 10)], 10, ('A', ['ACCC'], [0, 10])),                                  # :641
    ('deletion_insertion', [('ACCC', I, 10), ('ATGC', D, 11)], 10, ('ATGC', ['A', 'ACCCTGC'], [0, 11, 10])),   # :652
    ('two_deletions', [('AT', D, 10), ('ATGC', D, 11)], 10, ('ATGC', ['A', 'AGC'], [0, 11, 10])),    # :661
    ('two_insertions', [('AT', I, 10), ('ATGC', I, 11)], 10, ('A', ['AT', 'ATGC'], [0, 10, 11])),    # :670
    ('snp_deletion', [('C', S, 10), ('ATGC', D, 11)], 10, ('ATGC', ['A', 'CTGC'], [0, 11, 10])),     # :679
    ('snp_insertion', [('C', S, 10), ('ATGC', I, 11)], 10, ('A', ['ATGC', 'C'], [0, 11, 10])),       # :719
    ('kitchen_sink', [('C', S, 10), ('AA', I, 11), ('ACAC', I, 12), ('ATGC', D, 13), ('AT', D, 14)], 10,
     ('ATGC', ['A', 'AATGC', 'ACACTGC', 'AGC', 'CTGC'], [0, 13, 11, 12, 14, 10])),                   # :728
    ('min_count_rejects', [('C', S, 2), ('A', R, 10)], 3, None),                                     # :382
]


@pytest.mark.parametrize('name,alleles,min_count,expected', CALLER_KATS, ids=[k[0] for k in CALLER_KATS])
def test_caller_kats(tmp_path, name, alleles, min_count, expected):
  reads = _reads_for(alleles)
  ref = FakeRef([('chr1', SITE_REF)])
  kw = dict(vsc_min_count_snps=min_count, vsc_min_count_indels=min_count, vsc_min_fraction_snps=0.0, vsc_min_fraction_indels=0.0,
            sample_name='sample')
  table = _table(tmp_path, reads, [('chr1', SITE_REF)])
  got = [cand.canonical_call(r) for r in cand.candidates_in_region(table, ref, 'chr1', 10, 11, cand.CandidateOptions(**kw),
                                                                   rows=np.arange(table.n_reads)).records]
  want_oracle, _ = oc.candidates(SITE_REF, 'chr1', 10, 11, reads, oc.Options(
      min_count_snps=min_count, min_count_indels=min_count, min_fraction_snps=0.0, min_fraction_indels=0.0, sample_name='sample'))
  assert got == want_oracle
  if expected is None:
    assert got == []
    return
  ref_bases, alts, ad = expected
  assert len(got) == 1
  g = got[0]
  assert (g['ref'], g['alts'], g['info']['AD'], g['start'], g['end']) == (ref_bases, alts, ad, 10, 10 + len(ref_bases))
  assert g['info']['DP'] == [sum(ad)] and g['genotype'] == [-1, -1] and g['call_set_name'] == 'sample'
  assert g['info']['VAF'] == [a / sum(ad) for a in ad[1:]]
  for alt, n in zip(alts, ad[1:]):
    assert len(g['allele_support'][alt]) == n


def test_min_fraction_is_compared_as_float32(tmp_path):
  """VariantCallerOptions.min_fraction_snps is a proto float: 3 of 25 = 0.12 passes (double)0.12f = 0.1199999973."""
  reads = _reads_for([('C', S, 3), ('A', R, 22)])
  ref = FakeRef([('chr1', SITE_REF)])
  table = _table(tmp_path, reads, [('chr1', SITE_REF)])
  got = cand.candidates_in_region(table, ref, 'chr1', 10, 11, cand.CandidateOptions(), rows=np.arange(table.n_reads)).calls()
  assert len(got) == 1 and got[0].variant.alternate_bases == ['C']
  reads = _reads_for([('C', S, 3), ('A', R, 23)])      # 3 / 26 < 0.12
  table = _table(tmp_path, reads, [('chr1', SITE_REF)])
  assert cand.candidates_in_region(table, ref, 'chr1', 10, 11, cand.CandidateOptions(), rows=np.arange(table.n_reads)).records == []


def test_small_large_indel_fractions(tmp_path):
  """IndelAlleleFractionTest (variant_calling_multisample_test.cc:1192-1274): 100 reads, insertions AT x8, ATT x12, ATTT x6."""
  reads = _reads_for([('AT', I, 8), ('ATT', I, 12), ('ATTT', I, 6), ('A', R, 74)])
  ref = FakeRef([('chr1', SITE_REF)])
  table = _table(tmp_path, reads, [('chr1', SITE_REF)])
  base = dict(vsc_min_count_snps=1, vsc_min_count_indels=1, vsc_min_fraction_snps=0.0)
  o = cand.CandidateOptions(vsc_min_indel_fraction_for_small_indels=0.10, vsc_min_indel_fraction_for_large_indels=0.05,
                            vsc_small_indel_threshold=2, vsc_min_fraction_indels=0.0, **base)
  got = cand.candidates_in_region(table, ref, 'chr1', 10, 11, o, rows=np.arange(table.n_reads)).calls()
  assert sorted(len(a) for a in got[0].variant.alternate_bases) == [3, 4]          # ATT and ATTT kept, AT (8 %) dropped
  o = cand.CandidateOptions(vsc_min_indel_fraction_for_small_indels=0.10, vsc_min_indel_fraction_for_large_indels=0.05,
                            vsc_small_indel_threshold=0, vsc_min_fraction_indels=0.11, **base)
  got = cand.candidates_in_region(table, ref, 'chr1', 10, 11, o, rows=np.arange(table.n_reads)).calls()
  assert [len(a) for a in got[0].variant.alternate_bases] == [3]                    # threshold 0: min_fraction_indels decides


# ---- product == oracle on random inputs -----------------------------------------------------------------------------------
def _random_case(rng, n_reads, contig_len=200):
  contig = bytes(rng.choice(b'ACGTACGTACGTACGTN') for _ in range(contig_len))
  reads = []
  for i in range(n_reads):
    pos = rng.randrange(0, contig_len - 40)
    ops, seq, p = [], bytearray(), pos
    if rng.random() < 0.15:
      k = rng.randrange(1, 6)
      ops.append((4, k))
      seq += bytes(rng.choice(b'ACGT') for _ in range(k))
    if rng.random() < 0.05:
      k = rng.randrange(1, 4)
      ops.append((rng.choice([1, 2]), k))
      if ops[-1][0] == 1:
        seq += bytes(rng.choice(b'ACGT') for _ in range(k))
      else:
        p += k
    for _ in range(rng.randrange(1, 5)):
      k = rng.randrange(1, 30)
      ops.append((rng.choice([0, 0, 0, 7, 8]), k))
      for j in range(k):
        b = contig[p + j] if p + j < contig_len else ord('A')
        r = rng.random()
        seq.append(rng.choice(b'ACGT') if r < 0.08 or b == ord('N') else (ord('N') if r < 0.1 else b))
      p += k
      r = rng.random()
      k = rng.randrange(1, 5)
      if r < 0.25:
        ops.append((1, k))
        seq += bytes(rng.choice(b'ACGTN' if rng.random() < 0.1 else b'AC') for _ in range(k))
      elif r < 0.5:
        ops.append((2, k))
        p += k
      elif r < 0.55:
        ops.append((3, k))
        p += k
      if p >= contig_len + 20:
        break
    if ops[-1][0] in (2, 3) and rng.random() < 0.7:
      ops.append((0, 1))
      seq.append(contig[p] if p < contig_len else ord('A'))
    if rng.random() < 0.15:
      k = rng.randrange(1, 6)
      ops.append((4, k))
      seq += bytes(rng.choice(b'ACGT') for _ in range(k))
    merged = []
    for op, k in ops:        # adjacent equal ops are legal in BAM but keep the cigar tidy
      if merged and merged[-1][0] == op:
        merged[-1] = (op, merged[-1][1] + k)
      else:
        merged.append((op, k))
    quals = bytes(rng.choice([2, 8, 9, 10, 11, 25, 37, 40]) for _ in range(len(seq)))
    name = f'q{rng.randrange(0, n_reads // 2 + 1)}' if rng.random() < 0.2 else f'r{i}'      # repeated keys overwrite
    reads.append(protos.Read(fragment_name=name, read_number=0, position=pos, reverse_strand=rng.random() < 0.5,
                             mapping_quality=rng.choice([0, 3, 5, 20, 60]), cigar=merged, aligned_sequence=bytes(seq), aligned_quality=quals))
  return contig, reads


@pytest.mark.parametrize('seed', range(12))
def test_product_equals_oracle_on_random_reads(tmp_path, seed):
  rng = random.Random(1000 + seed)
  contig, reads = _random_case(rng, rng.choice([5, 120, 300]))
  ref = FakeRef([('chr1', contig)])
  table = _table(tmp_path, reads, [('chr1', contig)])
  assert table.n_reads == len(reads)
  start, end = rng.randrange(0, 50), rng.randrange(150, len(contig) + 1)
  mc = rng.choice([1, 2])
  kw = dict(min_mapping_quality=rng.choice([0, 5]), min_base_quality=10, track_ref_reads=seed % 2 == 1,
            small_model_vaf_context_window_size=rng.choice([0, 11, 51]), sample_name='s')
  legacy = seed % 5 == 4
  o = cand.CandidateOptions(vsc_min_fraction_multiplier=rng.choice([1.0, 0.5]), keep_legacy_allele_counter_behavior=legacy,
                            vsc_min_count_snps=mc, vsc_min_count_indels=mc, **kw)
  got = [cand.canonical_call(r) for r in cand.candidates_in_region(table, ref, 'chr1', start, end, o, rows=np.arange(len(reads))).records]
  want, counter = oc.candidates(contig, 'chr1', start, end, reads, oc.Options(
      min_fraction_multiplier=o.vsc_min_fraction_multiplier, keep_legacy_behavior=legacy, min_count_snps=mc, min_count_indels=mc, **kw))
  assert len(want) > 0 or len(reads) < 100
  assert got == want
  counts = cand.debug_allele_counts(table, ref, 'chr1', start, end, np.arange(len(reads)), o,
                                    [c['start'] for c in want] if o.track_ref_reads else [])
  for site, ac in zip(counts, counter.counts):
    assert site['ref'] == ac.ref_supporting_read_count
    assert sorted((a[3], a[0], a[1], a[2], a[4], a[5], a[6]) for a in site['alleles']) == sorted(
        (k, a['bases'], a['type'], int(a['low_quality']), a['mapq'], a['avg_bq'], int(a['reverse'])) for k, a in ac.read_alleles.items())


# ---- host helpers -----------------------------------------------------------------------------------------------------------
def test_regions_to_process_and_sharding():
  contigs = [('chr1', 2500), ('chr2', 900)]
  all_ = cand.regions_to_process(contigs, 1000)
  assert all_ == [('chr1', 0, 1000), ('chr1', 1000, 2000), ('chr1', 2000, 2500), ('chr2', 0, 900)]
  shards = [cand.regions_to_process(contigs, 1000, None, t, 3) for t in range(3)]
  assert sorted(sum(shards, [])) == sorted(all_) and shards[0] == [all_[0], all_[3]]
  assert cand.regions_to_process(contigs, 1000, ('chr1', 999, 2100)) == [('chr1', 999, 1999), ('chr1', 1999, 2100)]
  with pytest.raises(ValueError):
    cand.regions_to_process(contigs, 1000, None, 3, 3)
  with pytest.raises(ValueError):
    cand.regions_to_process(contigs, 1000, None, 1, None)


def test_reservoir_sample_matches_algorithm_r():
  """utils.reservoir_sample with a seeded RandomState: k of n retained, replaced slot j = randint(0, i + 1) < k."""
  got = cand.reservoir_sample(range(100), 10, np.random.RandomState(42))
  rs = np.random.RandomState(42)
  want = list(range(10))
  for i in range(10, 100):
    j = rs.randint(0, i + 1)
    if j < 10:
      want[j] = i
  assert got == want and len(set(got)) == 10
  assert cand.reservoir_sample(range(5), 10) == [0, 1, 2, 3, 4]
  with pytest.raises(ValueError):
    cand.reservoir_sample(range(5), -1)


def test_argument_errors(tmp_path):
  ref = FakeRef([('chr1', CHR1)])
  table = _table(tmp_path, [_read('r', 10, 'TCCGT', '5M')], [('chr1', CHR1)])
  from deepvariant_b200 import _lib
  with pytest.raises(_lib.DvbError):
    cand.candidates_in_region(table, ref, 'chr1', 20, 10, cand.CandidateOptions(), rows=np.arange(1))
  with pytest.raises(_lib.DvbError):
    cand.candidates_in_region(table, ref, 'chr1', 0, 10, cand.CandidateOptions(), rows=np.array([5]))


# ---- the reference's golden files ---------------------------------------------------------------------------------------------
def test_golden_fixture_candidates_reproduced(tmp_path):
  """Partitions of the reference's golden.calling_candidates whose reads the realigner left alone: every field of every
  DeepVariantCall (alleles, AD/DP/VAF, supporting read keys, per-read mapq / base quality / strand, VAF context)."""
  fx = json.load(open(os.path.join(GOLDEN, 'candidates_golden_subset.json')))
  contig = b'N' * fx['slice_start'] + fx['slice'].encode()
  contig += b'N' * (fx['n_bases'] - len(contig))
  ref = FakeRef([(fx['contig'], contig)])
  table = bam.NativeBamTable(os.path.join(GOLDEN, 'candidates_golden_subset.bam'), bam.ReadRequirements(min_mapping_quality=5))
  opts = cand.CandidateOptions(sample_name=fx['sample_name'], small_model_vaf_context_window_size=fx['small_model_vaf_context_window_size'])
  n = 0
  for part in fx['partitions']:
    got = [cand.canonical_call(r) for r in cand.candidates_in_region(table, ref, fx['contig'], part['start'], part['end'], opts).records]
    assert len(got) == len(part['expected'])
    for g, w in zip(got, part['expected']):
      w = dict(w)
      if not w.pop('af_exact'):
        g = dict(g, af_at_position=w['af_at_position'])
      assert g == w
      n += 1
  assert n >= 8


def test_pacbio_golden_variants_all_reproduced():
  """golden.pacbio_examples (realigner off) in chr20:9,060,000-9,065,000, from the reads of the reference's PacBio test BAM that overlap it
  (tests/golden/, tools/make_reference_subset_fixtures.py): 12 of 12 variants identical in site, alleles, AD, DP, VAF; none extra.
  All 341 of the whole 100 kb are pinned by tests/golden/candidates_golden_report.json."""
  sys.path.insert(0, os.path.join(ROOT, 'tools'))
  import check_candidates_golden as ck
  window = 'chr20_9060000_9065000'
  r = ck.pacbio_pin(os.path.join(GOLDEN, f'test_pacbio.{window}.bam'), os.path.join(GOLDEN, 'grch38.chr20_9030000_9135000.fa.gz'),
                    json.load(open(os.path.join(GOLDEN, f'golden.pacbio_variants.{window}.json'))), ('chr20', 9_060_000, 9_065_000))
  assert r['golden_variants'] == r['ours_candidates'] == r['identical_site_alleles_AD_DP_VAF'] == 12
  assert r['golden_only'] == r['ours_only'] == 0


def test_golden_report_is_current():
  r = json.load(open(os.path.join(GOLDEN, 'candidates_golden_report.json')))
  assert r['pacbio']['identical_site_alleles_AD_DP_VAF'] == r['pacbio']['golden_variants'] == 341
  assert r['golden_candidates'] == 78 and r['same_site_and_alleles'] >= 72 and r['identical_in_every_field'] >= 29


# ---- the make_examples stage CLI from --ref / --reads alone ----------------------------------------------------------------------
class OracleEncoder:
  """Stands in for pileup_image.GpuEncoder in the CPU run of the CLI test: same interface, pixels from the CPU oracle."""

  def __init__(self, params):
    import oracle_lib
    self.params, self._oracle = params, oracle_lib
    self.shape = (params.height, params.width, params.num_channels + params.num_alt_channels)

  def encode_host(self, batch):
    return self._oracle.encode_batch(self.params, batch)


def _planted_case(tmp_path):
  """A 6-kb genome, 40x of 100-bp paired reads, four planted variants (het SNP, hom SNP, het 2-bp insertion, het 3-bp deletion)."""
  rng = np.random.default_rng(5)
  n = 6000
  genome = ''.join(rng.choice(list('ACGT'), n))
  fa = tmp_path / 'ref.fa'
  fa.write_text('>chr20\n' + '\n'.join(genome[i:i + 60] for i in range(0, n, 60)) + '\n')
  (tmp_path / 'ref.fa.fai').write_text(f'chr20\t{n}\t7\t60\t61\n')
  snp_het, snp_hom, ins, dele = 1500, 2200, 3100, 3900
  recs = []
  for i in range(2000):
    pos = 1000 + int(rng.integers(0, 3900))
    hap = i % 2
    seq, cigar, p = [], [], pos
    run = 0
    while len(seq) < 100 and p < n - 10:
      if p == snp_hom or (p == snp_het and hap):
        seq.append('ACGT'[('ACGT'.index(genome[p]) + 1) % 4])
        run += 1
        p += 1
      elif p == ins and hap and run > 0:
        seq.append(genome[p])
        cigar += [(0, run + 1), (1, 2)]
        seq += ['G', 'T']
        run = 0
        p += 1
      elif p == dele and hap and run > 0:
        seq.append(genome[p])
        cigar += [(0, run + 1), (2, 3)]
        run = 0
        p += 4
      else:
        seq.append(genome[p])
        run += 1
        p += 1
    if run:
      cigar.append((0, run))
    if cigar[-1][0] != 0:
      continue
    merged = []
    for op, k in cigar:
      if merged and merged[-1][0] == op:
        merged[-1] = (op, merged[-1][1] + k)
      else:
        merged.append((op, k))
    seq = ''.join(seq)
    flag = 0x1 | 0x2 | (0x40 if i % 2 else 0x80) | (0x10 if i % 3 == 0 else 0)
    recs.append((pos, tb._record(0, pos, f'q{i}', 60, flag, merged, seq, rng.integers(20, 41, len(seq)).tolist(), 0, pos + 150, 250)))
  recs.sort(key=lambda t: t[0])
  bam_path = str(tmp_path / 'reads.bam')
  hdr_text = b'@HD\tVN:1.6\tSO:coordinate\n@RG\tID:rg\tSM:planted\n'
  hdr = b'BAM\1' + len(hdr_text).to_bytes(4, 'little') + hdr_text + (1).to_bytes(4, 'little') + (6).to_bytes(4, 'little') + b'chr20\0' + n.to_bytes(4, 'little')
  open(bam_path, 'wb').write(tb._bgzf(hdr + b''.join(r for _, r in recs)))
  return str(fa), bam_path, genome, dict(snp_het=snp_het, snp_hom=snp_hom, ins=ins, dele=dele)


def _run_cli(tmp_path, fa, bam_path, tag, realign=False, extra=()):
  from deepvariant_b200 import cli
  ex = str(tmp_path / f'{tag}.examples.tfrecord@1.gz')
  cands = str(tmp_path / f'{tag}.candidates.tfrecord.gz')
  assert cli.make_examples(['--mode', 'calling', '--ref', fa, '--reads', bam_path, '--examples', ex, '--candidates', cands,
                            '--channel_list', 'BASE_CHANNELS,insert_size', '--regions', 'chr20:1001-5000',
                            '--realign_reads' if realign else '--norealign_reads', *extra]) == 0
  from deepvariant_b200 import tfrecord
  return (list(tfrecord.read_records(str(tmp_path / f'{tag}.examples.tfrecord-00000-of-00001.gz'))), list(tfrecord.read_records(cands)))


def _check_planted(examples, cand_records, genome, sites):
  calls = [cand.canonical_call(r) for r in cand_records]
  by_start = {c['start']: c for c in calls}
  assert set(by_start) == set(sites.values())
  assert all(c['call_set_name'] == 'planted' for c in calls)                      # SM of the @RG line
  assert by_start[sites['snp_hom']]['info']['AD'][0] == 0
  het = by_start[sites['snp_het']]
  assert 0.3 < het['info']['VAF'][0] < 0.7 and len(het['alts']) == 1
  i = by_start[sites['ins']]
  assert i['ref'] == genome[sites['ins']] and i['alts'] == [genome[sites['ins']] + 'GT']
  d = by_start[sites['dele']]
  assert d['ref'] == genome[sites['dele']:sites['dele'] + 4] and d['alts'] == [genome[sites['dele']]]
  ex = [protos.parse_tf_example(r) for r in examples]
  assert len(ex) == 4 and [protos.parse_variant(e['variant/encoded'][1][0]).start for e in ex] == sorted(sites.values())
  assert all(e['image/shape'][1] == [100, 221, 7] for e in ex)
  # the examples carry the candidate's Variant (with AD / DP / VAF) byte for byte
  for e, c in zip(ex, cand_records):
    assert cand.canonical_call(protos.f_bytes(1, e['variant/encoded'][1][0]))['info'] == cand.canonical_call(c)['info']


def test_make_examples_cli_generates_candidates_cpu_plumbing(tmp_path, monkeypatch):
  """make_examples --ref --reads (no candidates file): regions -> reads -> allele counter -> caller -> pileups -> tf.Examples.
  The encoder is replaced by the CPU oracle here; the GPU twin below runs the product encoder and must give the same bytes."""
  from deepvariant_b200 import make_examples_native as men, pileup_image as pi
  monkeypatch.setattr(men.ExamplesGenerator, '_gpu', lambda self: OracleEncoder(pi.to_params(self.options.pic_options, height=self.pileup_image_height)))
  fa, bam_path, genome, sites = _planted_case(tmp_path)
  examples, cands = _run_cli(tmp_path, fa, bam_path, 'cpu')
  _check_planted(examples, cands, genome, sites)
  # with the realigner (the default): windows around the planted indels are assembled and their reads realigned; the planted
  # variants are clean, so the same four candidates come out, through the scratch-BAM / region-table path
  examples, cands = _run_cli(tmp_path, fa, bam_path, 'cpu_realigned', realign=True)
  _check_planted(examples, cands, genome, sites)
  # the VG Giraffe flag set (scripts/create_golden.sh:472-487): reads normalised after the realigner, legacy counter
  giraffe = ('--normalize_reads', '--keep_legacy_allele_counter_behavior', '--min_mapping_quality', '1')
  examples, cands = _run_cli(tmp_path, fa, bam_path, 'cpu_normalized', realign=True, extra=giraffe)
  _check_planted(examples, cands, genome, sites)
  examples, cands = _run_cli(tmp_path, fa, bam_path, 'cpu_normalized_only', realign=False, extra=giraffe)
  _check_planted(examples, cands, genome, sites)


# ---- the device pass, host-instantiated: dense counters, flags, exact calls on the flagged sites --------------------------------------
def _dense_from_counter(sites):
  """ref_count / substitution counts by base / other, derived from the host allele counter's entries (dvb_debug_allele_counts)."""
  n = len(sites)
  ref, subst, other, indel = np.zeros(n, np.int32), np.zeros((n, 4), np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8)
  for i, s in enumerate(sites):
    ref[i] = s['ref']
    for bases, typ, low, *_ in s['alleles']:
      if low:
        continue
      if typ == S:
        subst[i, 'ACGT'.index(bases)] += 1
      elif typ != R:
        other[i] += 1
        indel[i] |= typ in (I, D)
  return ref, subst, other, indel


def _check_device_pass_host_instantiation(table, ref, contig, start, end, rows, o):
  sites = cand.debug_allele_counts(table, ref, contig, start, end, rows, o)
  keys = [a[3] for s in sites for a in s['alleles']]
  unique_keys = all(len({a[3] for a in s['alleles']}) == len(s['alleles']) for s in sites) and len(set(
      table.names[int(table.name_begin[r]):int(table.name_begin[r + 1])] + bytes([table.read_number[r]]) for r in rows)) == len(rows)
  want_ref, want_subst, want_other, want_indel = _dense_from_counter(sites)
  for windowed in (False, True):
    counts, flags = cand.debug_dense_counts_host(table, ref, contig, start, end, rows, o, windowed=windowed)
    got_ref, got_subst, got_other = cand.split_dense_counts(counts, end - start)
    np.testing.assert_array_equal(got_ref, want_ref)          # ref_supporting_read_count is a plain counter in the reference too
    if unique_keys:                                           # a repeated read key is one map entry there, two counts here
      np.testing.assert_array_equal(got_subst, want_subst)
      np.testing.assert_array_equal(got_other, want_other)
      canon = np.frombuffer(ref._contig(contig)[start:end], np.uint8)
      canon = np.isin(canon, np.frombuffer(b'ACGT', np.uint8))
      np.testing.assert_array_equal((flags & 2) != 0, (want_indel != 0) & canon)      # no candidate on a non-ACGT reference base
  full = cand.candidates_in_region(table, ref, contig, start, end, o, rows=rows)
  starts = {cand.canonical_call(r)['start'] for r in full.records}
  flagged = set((np.nonzero(flags)[0] + start).tolist())
  if unique_keys:
    assert starts <= flagged                                  # the flags are a superset of the candidate sites
  if starts <= flagged:
    assert cand.candidates_at_flagged_positions(table, ref, contig, start, end, o, rows, flags).records == full.records
  return len(starts), len(flagged), len(keys)


@pytest.mark.parametrize('seed', range(8))
def test_device_pass_on_the_host_equals_the_allele_counter_random(tmp_path, seed):
  rng = random.Random(2000 + seed)
  contig, reads = _random_case(rng, rng.choice([120, 300]))
  if seed % 2 == 0:
    for i, r in enumerate(reads):
      r.fragment_name = f'u{i}'                               # unique keys: exact equality of every counter
  ref = FakeRef([('chr1', contig)])
  table = _table(tmp_path, reads, [('chr1', contig)])
  o = cand.CandidateOptions(min_mapping_quality=rng.choice([0, 5]), vsc_min_count_snps=rng.choice([1, 2]), vsc_min_count_indels=rng.choice([1, 2]),
                            small_model_vaf_context_window_size=rng.choice([0, 11]), keep_legacy_allele_counter_behavior=seed == 5, sample_name='s')
  n_c, n_f, _ = _check_device_pass_host_instantiation(table, ref, 'chr1', rng.randrange(0, 50), rng.randrange(150, len(contig) + 1),
                                                      np.arange(len(reads)), o)
  assert n_c > 0 and n_f >= n_c


def test_device_pass_on_the_host_on_the_golden_fixture():
  fx = json.load(open(os.path.join(GOLDEN, 'candidates_golden_subset.json')))
  contig = b'N' * fx['slice_start'] + fx['slice'].encode()
  contig += b'N' * (fx['n_bases'] - len(contig))
  ref = FakeRef([(fx['contig'], contig)])
  table = bam.NativeBamTable(os.path.join(GOLDEN, 'candidates_golden_subset.bam'), bam.ReadRequirements(min_mapping_quality=5))
  o = cand.CandidateOptions(sample_name=fx['sample_name'], small_model_vaf_context_window_size=51)
  for part in fx['partitions']:
    rows = cand.region_reads(table, fx['contig'], part['start'], part['end'])
    n_c, n_f, _ = _check_device_pass_host_instantiation(table, ref, fx['contig'], part['start'], part['end'], rows, o)
    assert n_c == len(part['expected']) and n_f < 0.1 * (part['end'] - part['start'])      # the pre-filter is selective


def test_gpu_allele_counter_needs_a_device(tmp_path):
  import torch
  if torch.cuda.is_available():
    pytest.skip('a CUDA device is present')
  from deepvariant_b200 import _lib
  table = _table(tmp_path, [_read('r', 10, 'TCCGT', '5M')], [('chr1', CHR1)])
  with pytest.raises(_lib.DvbError, match='no CUDA device'):
    cand.GpuAlleleCounter(table)


def test_make_examples_cli_windowed_reads_equal_the_whole_table(tmp_path, monkeypatch):
  """Without --regions the reads are held one genome window at a time (DVB_READ_WINDOW_BP; the default when the file has an index):
  the same examples and candidates as with every read resident, windows smaller than the spacing of the planted variants, with and
  without the realigner, and for two tasks of a sharded run."""
  from deepvariant_b200 import cli, make_examples_native as men, pileup_image as pi, tfrecord
  monkeypatch.setattr(men.ExamplesGenerator, '_gpu', lambda self: OracleEncoder(pi.to_params(self.options.pic_options, height=self.pileup_image_height)))
  fa, bam_path, genome, sites = _planted_case(tmp_path)

  def run(tag, window, extra=()):
    if window:
      monkeypatch.setenv('DVB_READ_WINDOW_BP', str(window))
    else:
      monkeypatch.delenv('DVB_READ_WINDOW_BP', raising=False)
    ex = str(tmp_path / f'{tag}.examples.tfrecord.gz')
    cands = str(tmp_path / f'{tag}.candidates.tfrecord.gz')
    assert cli.make_examples(['--mode', 'calling', '--ref', fa, '--reads', bam_path, '--examples', ex, '--candidates', cands,
                              '--channel_list', 'BASE_CHANNELS,insert_size', *extra]) == 0
    return list(tfrecord.read_records(ex)), list(tfrecord.read_records(cands))
  for extra in (('--norealign_reads',), ('--realign_reads',), ('--norealign_reads', '--gvcf', str(tmp_path / 'g.tfrecord.gz'))):
    whole = run('whole', 0, extra)
    assert len(whole[0]) == 4
    for window in (1000, 1700, 100000):
      assert run(f'w{window}', window, extra) == whole
  # two tasks of a sharded run: each walks its own partitions (every second kilobase) across the windows
  shards = {}
  for window in (0, 1000):
    if window:
      monkeypatch.setenv('DVB_READ_WINDOW_BP', str(window))
    else:
      monkeypatch.delenv('DVB_READ_WINDOW_BP', raising=False)
    for task in range(2):
      assert cli.make_examples(['--mode', 'calling', '--ref', fa, '--reads', bam_path, '--examples', str(tmp_path / f's{window}.tfrecord@2.gz'),
                                '--channel_list', 'BASE_CHANNELS,insert_size', '--norealign_reads', '--task', str(task)]) == 0
    shards[window] = [list(tfrecord.read_records(str(tmp_path / f's{window}.tfrecord-0000{t}-of-00002.gz'))) for t in range(2)]
  assert shards[0] == shards[1000] and sum(len(x) for x in shards[0]) == 4
