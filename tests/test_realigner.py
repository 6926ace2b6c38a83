"""Local realigner (deepvariant_b200/realigner.py): window selector, de Bruijn graph, assembly + FastPassAligner.

Known answers transcribed from deepvariant/realigner/window_selector_test.py:455-540 and python/debruijn_graph_wrap_test.py:80-360;
the reference's WGS goldens - made WITH the realigner - end to end from the reads of its NA12878 test BAM that start before
chr20:10,011,000 (tests/golden/, tools/make_reference_subset_fixtures.py): 78 of 78 golden candidates identical in every field and 84 of
84 golden.calling_examples images byte for byte (tools/check_realigner_golden.py).  CPU-only."""
import json
import os
import sys

import pytest

from deepvariant_b200 import realigner as rl
from deepvariant_b200.protos import Read

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
# the reference bases of chr20:9,990,000-10,020,000, where the reads of the window BAM lie
QUICKSTART_FASTA = os.path.join(GOLDEN, 'quickstart.chr20_10mb.fa.gz')


def _read(seq, pos=1, qual=30, mapq=60):
  return Read(fragment_name='read', position=pos, mapping_quality=mapq, cigar=[(0, len(seq))], aligned_sequence=seq.encode(),
              aligned_quality=bytes([qual] * len(seq)))


def _single_k(k):
  return rl.DeBruijnGraphOptions(min_k=k, max_k=k, step_k=1, min_mapq=14, min_base_quality=15, min_edge_weight=2, max_num_paths=256)


def test_debruijn_graph_basics_and_pruning():
  ref, read = 'GATTACA', 'GATGACA'
  g = rl.build_graph(ref, [_read(read), _read(read)], _single_k(3))                      # test_basics: two reads keep the read path
  assert sorted(g.candidate_haplotypes()) == sorted([ref, read])
  edges = {(a, b): tuple(e) for a, ws in g.out.items() for b, e in ws.items()}
  assert edges == {('GAT', 'ATT'): (1, True), ('ATT', 'TTA'): (1, True), ('TTA', 'TAC'): (1, True), ('TAC', 'ACA'): (1, True),
                   ('GAT', 'ATG'): (2, False), ('ATG', 'TGA'): (2, False), ('TGA', 'GAC'): (2, False), ('GAC', 'ACA'): (2, False)}
  g = rl.build_graph(ref, [_read(read)], _single_k(3))                                   # test_pruning_1: one read is pruned away
  assert g.candidate_haplotypes() == [ref] and list(g.out) == ['GAT', 'ATT', 'TTA', 'TAC', 'ACA']
  assert rl.build_graph('GATTACATG', [_read(read), _read(read)], _single_k(8)) is not None    # test_k_exceeds_read_length
  assert rl.build_graph(ref, [], _single_k(7)) is None and rl.build_graph(ref, [], _single_k(8)) is None   # test_k_exceeds_ref_length
  low = _read(read, qual=10)                                                              # bases under min_base_quality add no edges
  assert rl.build_graph(ref, [low, low], _single_k(3)).candidate_haplotypes() == [ref]
  assert rl.build_graph(ref, [_read(read, mapq=5)] * 2, _single_k(3)).candidate_haplotypes() == [ref]


@pytest.mark.parametrize('ref,smallest_good_k', [
    ('ACGTACGT', 5), ('ACGTAAACGT', 5), ('ACGTAAACGTAAA', 8), ('AAACGTAAACGT', 7), ('AAACGTAAACGTAAA', 10),
    ('TGGTAAGTTTATAAGGTTATAAGCTGAGAGGTTTTGCTGATCTTGGCTGAGCTCAGCTGGGCAGGTCTTCCGGTCTTGGCTGGGGTTCACTGACACACAAGCAGCTGACAGTTGGCTGATCTAGGATGGCCTCAGCTGGG', 11),
])
def test_reference_cycle_detector(ref, smallest_good_k):
  for k in range(max(smallest_good_k - 5, 1), min(smallest_good_k + 5, len(ref))):
    assert (rl.build_graph(ref, [], _single_k(k)) is None) == (k < smallest_good_k), k


@pytest.mark.parametrize('candidates,expected', [
    ([100, 200, 300], [(96, 104), (196, 204), (296, 304)]), ([2, 8], [(-2, 12)]), ([2, 14], [(-2, 6), (10, 18)]),
    ([2, 10], [(-2, 14)]), ([2, 11], [(-2, 6), (7, 15)]), ([], []),
])
def test_candidates_to_windows(candidates, expected):
  assert rl.candidates_to_windows(candidates, rl.WindowSelectorOptions(min_windows_distance=4)) == expected


def test_variant_reads_candidate_positions():
  """VariantReadsWindowSelectorCandidates (window_selector.cc:85-125): substitutions count at their position, insertions / soft
  clips over [i + 1 - len, i + len), deletions over (i, i + len]; alleles seen in fewer than two reads are ignored."""
  def site(ref, *alleles):
    return {'ref': ref, 'alleles': [[b, t, 0, f'r{k}', 60, 30, 0] for k, (b, t) in enumerate(alleles)]}
  sites = [site(5)] * 3 + [site(3, ('C', 2), ('C', 2))] + [site(5)] * 3 + [site(3, ('ATT', 3), ('ATT', 3), ('G', 2))] + [site(5)] * 3 + \
          [site(4, ('CAA', 4), ('CAA', 4))] + [site(5)] * 4
  o = rl.WindowSelectorOptions()
  got = rl.candidate_positions_from_counts(sites, 1000, o)
  assert got == [1003] + [1006, 1007, 1008, 1009] + [1012, 1013]


def test_wgs_goldens_made_with_the_realigner_are_reproduced_end_to_end():
  sys.path.insert(0, os.path.join(ROOT, 'tools'))
  import check_realigner_golden
  r = check_realigner_golden.main(td=GOLDEN, bam_path=os.path.join(GOLDEN, 'NA12878_S1.chr20.10_10p1mb.window.bam'), ref_path=QUICKSTART_FASTA,
                                  shard_keys=json.load(open(os.path.join(GOLDEN, 'golden.calling_examples.shard_keys.json'))), write=False)
  assert r['golden_candidates'] == r['ours_candidates'] == r['candidates_identical_in_every_field'] == 78
  assert r['golden_examples'] == r['examples_planned'] == r['images_identical'] == 84
  assert r['golden_read_rows'] == r['golden_read_rows_reproduced'] == 4309
  # the tf.Examples themselves (assertDeepVariantExamplesEqual: every feature decoded), their order, and --task i of 3 sharding
  assert r['tf_examples_equal_feature_by_feature'] == 84 and r['example_order_equal'] and r['sharded_goldens_equal_task_by_task'] == [True] * 3


def test_realigner_report_is_committed():
  r = json.load(open(os.path.join(ROOT, 'tests/golden/realigner_golden_report.json')))
  assert r['candidates_identical_in_every_field'] == 78 and r['images_identical'] == 84


def test_wgs_alt_aligned_goldens_diff_channels_and_rows():
  """golden.alt_aligned_pileup_{diff_channels,rows}_examples: 49 of 49 images each (100 x 221 x 8 / 300 x 221 x 6), realigner on;
  the golden images are held as SHA-256 digests (golden.alt_aligned_pileup.digests.json)."""
  sys.path.insert(0, os.path.join(ROOT, 'tools'))
  import check_alt_aligned_wgs_golden
  digests = json.load(open(os.path.join(GOLDEN, 'golden.alt_aligned_pileup.digests.json')))
  for layout in ('diff_channels', 'rows'):
    r = check_alt_aligned_wgs_golden.run(layout, digests[layout], os.path.join(GOLDEN, 'NA12878_S1.chr20.10_10p1mb.window.bam'), QUICKSTART_FASTA)
    assert r['compared'] == r['images_identical'] == r['golden_examples'] == 49 and r['of_those_identical'] == r['examples_with_alt_aligned_pileups'] == 4


def test_rows_and_single_row_composition():
  import numpy as np
  from deepvariant_b200 import make_examples_native as men, pileup_image as pi
  pic = pi.default_options()
  imgs = np.arange(5 * 4 * 3 * 2, dtype=np.uint8).reshape(5, 4, 3, 2)       # 2 plans + 3 alt-aligned pileups, H = 4
  pic.alt_aligned_pileup = 'rows'
  out = men.compose_alt_aligned(imgs, 2, [[2, 3], [4]], pic, [['A', 'AT'], ['G']])
  assert out.shape == (2, 12, 3, 2)
  assert np.array_equal(out[0, :4], imgs[0]) and np.array_equal(out[0, 4:8], imgs[2]) and np.array_equal(out[0, 8:], imgs[3])
  assert np.array_equal(out[1, 4:8], imgs[4]) and not out[1, 8:].any()       # a single alt: the third section stays blank
  pic.alt_aligned_pileup = 'single_row'
  out = men.compose_alt_aligned(imgs, 2, [[2, 3], [4]], pic, [['A', 'AT'], ['G']])
  assert out.shape == (2, 8, 3, 2) and np.array_equal(out[0, 4:], imgs[3]) and np.array_equal(out[1, 4:], imgs[4])   # the longer alt's pileup
  out = men.compose_alt_aligned(imgs, 2, [[2, 3], []], pic, [['AT', 'A'], ['G']])
  assert np.array_equal(out[0, 4:], imgs[2]) and not out[1, 4:].any()


def test_native_de_bruijn_graph_equals_python_restatement():
  """csrc/dvb_dbg.cu (dvb_dbg_candidate_haplotypes) against DeBruijnGraph / build_graph on random windows: repeats in the
  reference (k search, cycles), reads with substitutions / insertions / N / low qualities / low mapping quality / lower case,
  path-count overflow; the three outcomes (no graph, a graph without a path, haplotypes) all occur."""
  import numpy as np
  rng = np.random.default_rng(1)
  outcomes = {'none': 0, 'empty': 0, 'ref_only': 0, 'several': 0}
  for trial in range(400):
    n = int(rng.integers(30, 300))
    ref = ''.join(rng.choice(list('ACGT'), n))
    if trial % 5 == 0:
      ref = ref[:n // 2] + ref[:n // 2]
      n = len(ref)
    snps = sorted(set(int(x) for x in rng.integers(5, n - 5, int(rng.integers(0, 6)))))       # planted on haplotype 1
    ins_at = int(rng.integers(5, n - 5))                                                       # planted on haplotype 2
    reads = []
    for i in range(int(rng.integers(0, 80))):
      s, length = int(rng.integers(0, max(1, n - 20))), int(rng.integers(25, 120))
      seq = []
      for pos in range(s, min(n, s + length)):
        b = ref[pos]
        if i % 3 == 1 and pos in snps:
          b = 'ACGT'[('ACGT'.index(b) + 1) % 4]
        seq.append(b)
        if i % 3 == 2 and pos == ins_at:
          seq += list('GATTACA')
      for j in range(len(seq)):
        if rng.random() < 0.004:
          seq[j] = 'N'
      seq = ''.join(seq)
      if rng.random() < 0.1:
        seq = seq.lower()
      quals = bytes(rng.choice([5, 20, 30, 40, 40, 40, 40, 40, 40, 40, 40, 40], len(seq)).astype(np.uint8))
      reads.append(Read(fragment_name=f'r{i}', aligned_sequence=seq.encode(), aligned_quality=quals, mapping_quality=int(rng.choice([5, 20, 60, 60]))))
    o = rl.DeBruijnGraphOptions(min_k=int(rng.choice([3, 6, 10])), max_k=int(rng.choice([12, 30, 101])), step_k=int(rng.choice([1, 2])),
                                max_num_paths=int(rng.choice([4, 256])))
    g = rl.build_graph(ref, reads, o)
    want = None if g is None else g.candidate_haplotypes()
    got = rl.candidate_haplotypes_native(ref, reads, o)
    assert got == want, (trial, o)
    outcomes['none' if want is None else 'empty' if not want else 'ref_only' if want == [ref] else 'several'] += 1
  assert all(v > 5 for v in outcomes.values()), outcomes
