"""End-to-end pin of the PACBIO make_examples path against the reference's golden.pacbio_examples.tfrecord.gz (401 examples,
100 x 147 x 10; make_examples_test.py:792-831: realigner off, --track_ref_reads, --phase_reads, --sort_by_haplotypes,
--trim_reads_for_pileup, --alt_aligned_pileup diff_channels, --partition_size 25000, --min_mapping_quality 1).

For every 25-kb partition: region reads -> candidates over the padded region (csrc/dvb_candidates.cu) -> direct phasing
(deepvariant_b200/direct_phasing.py) -> HP on the reads -> trimmed pileups through the planner + CPU oracle, compared with the golden
images on the seven computed channels (read_base, base_quality, mapping_quality, strand, read_supports_variant,
base_differs_from_ref, haplotype): whole image, row order included.  base_methylation (channel 7) is all zero in the golden; the two
alt-aligned channels (haplotype realignment: FastPassAligner + Smith-Waterman, SURVEY 8(f) #3) are compared too.
Writes tests/golden/pacbio_end_to_end_report.json."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_lib  # noqa: E402
from deepvariant_b200 import bam, candidates as cand, direct_phasing, fasta, packing, protos, tfrecord  # noqa: E402
from deepvariant_b200 import make_examples_native as men  # noqa: E402
from deepvariant_b200 import pileup_image as pi  # noqa: E402

T = '/root/reference/deepvariant/testdata/'
REGION = ('chr20', 8999999, 9100000)


def channel_summary(img: np.ndarray) -> dict:
  """Per channel of an example image: SHA-256 of its pixels and whether any is set; and its non-blank read rows."""
  from check_alt_aligned_wgs_golden import image_digest
  chans = [np.ascontiguousarray(img[..., c]) for c in range(img.shape[-1])]
  return {'digests': [image_digest(c.tobytes(), c.shape) for c in chans], 'nonzero': [bool(c.any()) for c in chans],
          'rows': int(sum(1 for r in range(5, img.shape[0]) if img[r].any()))}


def golden_summaries(path: str) -> list:
  """[start, alt allele indices, channel_summary] per example of a golden examples file."""
  out = []
  for r in tfrecord.read_records(path):
    e = protos.parse_tf_example(r)
    img = np.frombuffer(e['image/encoded'][1][0], dtype=np.uint8).reshape(e['image/shape'][1])
    out.append([protos.parse_variant(e['variant/encoded'][1][0]).start, protos.parse_alt_allele_indices(e['alt_allele_indices/encoded'][1][0]),
                channel_summary(img)])
  return out


def main(bam_path=None, ref_path=None, golden=None, region=REGION, write=True):
  """golden: golden_summaries of the examples to compare with (default: all of the testdata's golden.pacbio_examples); region: the
  part of chr20 to make examples for, in 25-kb partitions from its start.  Returns the stats."""
  if golden is None:
    golden = golden_summaries(T + 'golden.pacbio_examples.tfrecord.gz')
  golden = {(start, tuple(idx)): g for start, idx, g in golden}
  bam_path = bam_path or T + 'input/test_pacbio.chr20_100kbp_at_9mb.bam'
  table = bam.NativeBamTable(bam_path, bam.ReadRequirements(min_mapping_quality=1), parse_aux=True)
  ref = fasta.IndexedFastaReader(ref_path or T + 'input/grch38.chr20_and_21_10M.fa.gz')
  copts = cand.CandidateOptions(sample_name=cand.sample_name_from_bam(bam_path), min_mapping_quality=1, track_ref_reads=True,
                                vsc_min_fraction_indels=0.12, partition_size=25000)
  pic = pi.default_options(pi.ReadRequirements(min_base_quality=10, min_mapping_quality=1))
  pic.channels = pi.PILEUP_DEFAULT_CHANNELS + ['haplotype', 'base_methylation', 'diff_channels_alternate_allele_1', 'diff_channels_alternate_allele_2']   # the golden's own ten channels [1-7, 23, 9, 10]; the test BAM has no MM / ML tags, so base_methylation is all zero
  pic.num_channels = len(pic.channels)
  pic.alt_aligned_pileup = 'diff_channels'
  pic.width = 147
  pic.sort_by_haplotypes = True
  gen = men.ExamplesGenerator(men.MakeExamplesOptions(pic_options=pic, trim_reads_for_pileup=True), test_mode=True, ref_reader=ref)
  params = pi.to_params(pic)
  stats = dict(examples=0, images_equal_7_channels=0, haplotype_channel_equal=0, row_order_equal=0, reads_phased=0, reads=0, snp_examples=0,
               snp_alt_aligned_channels_zero_in_golden=0, methylation_channel_zero=0)
  mismatches = []
  for contig, s, e in cand.regions_to_process([(c, ref.n_bases(c)) for c in ref.contig_order], 25000, region):
    rows = cand.region_reads(table, contig, s, e, copts.max_reads_per_partition, copts.random_seed)
    found = cand.candidates_in_region(table, ref, contig, s, e, copts, rows=rows, padding_pct=20)
    reads = [table.read(int(r)) for r in rows]                      # fresh Read objects for this region, like a new BAM query
    phases = direct_phasing.phase_reads([cand.canonical_call(r) for r in found.all_records], [r.key() for r in reads])
    for r, p in zip(reads, phases):
      r.hp_values = [p]
    stats['reads'] += len(reads)
    stats['reads_phased'] += sum(1 for p in phases if p)
    plans = gen.plan_region(found.calls(), reads, {})
    if not plans:
      continue
    specs, alt_at = [p.spec for p in plans], []
    for p in plans:
      alt_at.append(list(range(len(specs), len(specs) + len(p.alt_specs))))
      specs += p.alt_specs
    ours = men.compose_alt_aligned(oracle_lib.encode_batch(params, packing.pack_images(specs, params)), len(plans), alt_at, pic)
    for p, img in zip(plans, ours):
      idx = tuple(p.variant.alternate_bases.index(a) for a in p.alt_combination)
      g = golden.get((p.variant.start, idx))
      if g is None:
        mismatches.append({'start': p.variant.start, 'why': 'not in golden'})
        continue
      o = channel_summary(img)
      same = [a == b for a, b in zip(o['digests'], g['digests'])]
      stats['examples'] += 1
      eq7 = all(same[:7])
      stats['images_equal_7_channels'] += eq7
      stats['haplotype_channel_equal'] += same[6]
      stats['row_order_equal'] += all(same[:4])
      stats['methylation_channel_zero'] += not g['nonzero'][7]
      alt_eq = all(same[8:10])
      stats['alt_aligned_channels_equal'] = stats.get('alt_aligned_channels_equal', 0) + alt_eq
      stats['whole_image_equal'] = stats.get('whole_image_equal', 0) + all(same)   # all ten channels, the golden's own layout
      if p.variant_type != 1:
        stats['indel_examples'] = stats.get('indel_examples', 0) + 1
        stats['indel_alt_aligned_channels_equal'] = stats.get('indel_alt_aligned_channels_equal', 0) + alt_eq
        if not alt_eq and len(mismatches) < 40:
          mismatches.append({'start': p.variant.start, 'alts': p.alt_combination, 'alt_channels_differ': [c for c in (8, 9) if not same[c]],
                             'rows': g['rows']})
      if p.variant_type == 1:
        stats['snp_examples'] += 1
        stats['snp_alt_aligned_channels_zero_in_golden'] += not any(g['nonzero'][8:])
      if not eq7 and len(mismatches) < 40:
        mismatches.append({'start': p.variant.start, 'alts': p.alt_combination, 'channels_differ': [c for c in range(7) if not same[c]],
                           'rows_ours': o['rows'], 'rows_golden': g['rows']})
  stats['golden_examples'] = len(golden)
  if write:
    print(json.dumps(stats, indent=1))
    print(json.dumps(mismatches[:10], indent=1))
    with open(os.path.join(ROOT, 'tests/golden/pacbio_end_to_end_report.json'), 'w') as f:
      json.dump({'stats': stats, 'first_mismatches': mismatches}, f, indent=1)
  return stats


if __name__ == '__main__':
  main()
