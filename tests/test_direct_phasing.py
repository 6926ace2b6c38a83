"""Direct phasing (deepvariant_b200/direct_phasing.py) against the known-answer tests of deepvariant/direct_phasing_test.cc:491-965
(transcribed as data; min_alleles_to_phase = 2 as in CreateDefaultDirectPhasing) and end to end against the reference's golden PACBIO
examples of one 25-kb partition (candidates -> phasing -> haplotype-sorted pileups, every image).  CPU-only."""
import json
import os
import sys

import pytest

from deepvariant_b200 import direct_phasing as dp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cand(start, end, support, ref_support=()):
  ext = lambda names: [{'read_name': n, 'is_low_quality': 0} for n in names]
  return {'start': start, 'end': end, 'alts': sorted(support), 'allele_support_ext': {a: ext(v) for a, v in support.items()},
          'ref_support_ext': ext(ref_support)}


def _reads(n):
  return [f'read{i}/0' for i in range(1, n + 1)]


def _r(*idx):
  return [f'read{i}/0' for i in idx]


KATS = [
    ('simple', [(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5)}), (105, 106, {'C': _r(1, 2, 4, 5)}), (110, 111, {'T': _r(1, 2, 3), 'G': _r(4, 5)})],
     5, [1, 1, 1, 2, 2]),                                                                                                       # :491
    ('error_correction', [(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5)}), (105, 106, {'C': _r(1, 2, 3, 4, 5)}),
                          (110, 111, {'T': _r(1, 2), 'G': _r(3, 4, 5)}), (120, 121, {'T': _r(1, 2, 3), 'G': _r(4, 5)})], 5, [1, 1, 1, 2, 2]),   # :521
    ('changed_order_of_alleles', [(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5)}), (105, 106, {'C': _r(1, 2, 3, 4, 5)}),
                                  (110, 111, {'T': _r(4, 5), 'G': _r(1, 2, 3)}), (120, 121, {'G': _r(4, 5), 'T': _r(1, 2, 3)})], 5, [1, 1, 1, 2, 2]),   # :558
    ('unphased_read', [(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5)}), (105, 106, {'C': _r(1, 2, 3, 4, 5)}),
                       (110, 111, {'T': _r(1, 2), 'G': _r(4, 5, 3)})], 5, [1, 1, 0, 2, 2]),                                 # :597
    ('broken_path', [(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5)}), (105, 106, {'C': _r(4, 5), 'G': _r(6, 7)}),
                     (110, 111, {'T': _r(6, 7), 'G': _r(4, 5)})], 7, [0, 0, 0, 2, 2, 1, 1]),                                # :630
    ('fully_connected', [(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5, 6)}), (105, 106, {'C': _r(4, 5, 1), 'G': _r(2, 3, 6)}),
                         (110, 111, {'T': _r(1, 2, 3), 'G': _r(4, 5, 6)})], 6, [1, 1, 1, 2, 2, 2]),                          # :822
    ('two_blocks_with_score_tie', [(100, 101, {'A': _r(1, 2), 'C': _r(3, 4)}), (110, 111, {'G': _r(1, 2), 'T': _r(3, 4)}),
                                   (120, 121, {'A': _r(5, 6, 7, 8), 'C': _r(9, 10, 11, 12)})], 12, [1, 1, 2, 2, 0, 0, 0, 0, 0, 0, 0, 0]),   # :913
]


@pytest.mark.parametrize('name,cands,n_reads,expected', KATS, ids=[k[0] for k in KATS])
def test_phase_reads_kats(name, cands, n_reads, expected):
  got = dp.phase_reads([_cand(*c) for c in cands], _reads(n_reads), min_alleles_to_phase=2)
  assert got == expected


def test_unordered_candidates_are_rejected():
  """PhaseReadUnorderedInputFail / PhaseReadCandidateOutOfOrderInTheMiddle (:853-911): the reference CHECK-fails."""
  cands = [_cand(105, 106, {'C': _r(4, 5, 1), 'G': _r(2, 3, 6)}), _cand(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5, 6)})]
  with pytest.raises(ValueError):
    dp.phase_reads(cands, _reads(6))


def test_candidate_filter_and_low_quality_support():
  """FilterOneAlleleCandidate / FilterCandidateWithIndel (:967-1030) and ReadSupportFromProtoLQReads (:210-241)."""
  # one called allele and fewer than three reference reads: not phasable -> nobody is phased
  cands = [_cand(100, 101, {'A': _r(1, 2, 3)}), _cand(105, 106, {'C': _r(1, 2, 3)})]
  assert dp.phase_reads(cands, _reads(3)) == [0, 0, 0]
  # an indel candidate is skipped, and so is the SNP inside its span
  cands = [_cand(100, 101, {'A': _r(1, 2, 3), 'C': _r(4, 5, 6)}), _cand(102, 106, {'G': _r(1, 2, 3), 'GTTTT': _r(4, 5, 6)}),
           _cand(104, 105, {'T': _r(1, 2, 3), 'G': _r(4, 5, 6)}), _cand(110, 111, {'T': _r(1, 2, 3), 'G': _r(4, 5, 6)})]
  d = dp.DirectPhasing()
  assert d.phase(cands, _reads(6)) == [1, 1, 1, 2, 2, 2] and d.positions == [100, 110]
  # low-quality support and reads that are not in the region do not enter the graph
  c = _cand(100, 101, {'A': _r(1, 2, 9), 'C': _r(3, 4)})
  c['allele_support_ext']['A'][0]['is_low_quality'] = 1
  d = dp.DirectPhasing()
  d.phase([c], _reads(4))
  assert sorted(s.read_index for s in d.vertices[0].read_support) == [1]
  # a reference vertex needs three supporting reads
  c = _cand(100, 101, {'A': _r(1, 2)}, ref_support=_r(3, 4, 5))
  d = dp.DirectPhasing()
  d.phase([c, _cand(105, 106, {'C': _r(1, 2)}, ref_support=_r(3, 4, 5))], _reads(5))
  assert [v.bases for v in d.vertices] == ['REF', 'A', 'REF', 'C'] and d.phase([c], _reads(5)) == [0] * 5
  assert dp.phase_reads([_cand(100 + i, 101 + i, {'A': _r(1)}) for i in range(3)], _reads(2), phase_max_candidates=2) == [0, 0]


def test_pacbio_golden_examples_end_to_end():
  """candidates -> direct phasing -> trimmed, haplotype-sorted pileups == the reference's golden.pacbio_examples on the seven
  computed channels, row order included, AND on the two alt-aligned diff channels, for all 126 examples of its partition
  chr20:9,074,999-9,099,999 (the golden's base_methylation channel is all zero).  The inputs are the reads of its PacBio test BAM
  overlapping the padded partition, byte for byte; the golden images are held as per-channel SHA-256 digests (tests/golden/,
  tools/make_reference_subset_fixtures.py).  All 401 examples of the 100 kb are pinned by the committed report below."""
  sys.path.insert(0, os.path.join(ROOT, 'tools'))
  import check_pacbio_end_to_end
  g = os.path.join(ROOT, 'tests', 'golden')
  golden = json.load(open(os.path.join(g, 'golden.pacbio_examples.chr20_9074999_9099999.json')))
  s = check_pacbio_end_to_end.main(os.path.join(g, 'test_pacbio.chr20_9074999_9099999.bam'), os.path.join(g, 'grch38.chr20_9030000_9135000.fa.gz'),
                                   golden, ('chr20', 9_074_999, 9_099_999), write=False)
  n = len(golden)
  assert s['examples'] == s['golden_examples'] == s['images_equal_7_channels'] == s['haplotype_channel_equal'] == s['whole_image_equal'] == n == 126
  assert s['snp_examples'] == s['snp_alt_aligned_channels_zero_in_golden'] and s['methylation_channel_zero'] == n
  # alt-aligned pileups (FastPassAligner + Smith-Waterman against each alt haplotype): every indel example's two diff channels
  assert s['indel_examples'] == s['indel_alt_aligned_channels_equal'] > 0 and s['snp_examples'] + s['indel_examples'] == n
  assert s['reads_phased'] > 0


def test_end_to_end_report_is_committed():
  s = json.load(open(os.path.join(ROOT, 'tests/golden/pacbio_end_to_end_report.json')))['stats']
  assert s['images_equal_7_channels'] == s['whole_image_equal'] == s['golden_examples'] == 401
