"""Pins candidate generation (csrc/dvb_candidates.cu) against the reference's golden candidates.

Runs where /root/reference exists.  Re-derives golden.calling_candidates.tfrecord.gz (78 DeepVariantCalls; make_examples
--regions chr20:10,000,000-10,010,000 on NA12878_S1.chr20.10_10p1mb.bam, scripts/create_golden.sh:165-176) from the raw BAM
with our allele counter + caller and compares, per candidate: reference / alternate bases, AD / DP / VAF, allele_support as sets
of read keys, allele_support_ext (mapping quality, average base quality, strand, low-quality flag per read) and
allele_frequency_at_position.  The golden was made with the realigner on, so candidates whose reads the realigner rewrote are
expected to differ; the report lists them.  Writes tests/golden/candidates_golden_report.json and a fixture of the candidates
that match (tests/golden/candidates_golden_subset.json) used by tests/test_candidates.py where the reference is absent.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deepvariant_b200 import bam, candidates as cand, fasta, protos, tfrecord  # noqa: E402

canonical = cand.canonical_call

TESTDATA = '/root/reference/deepvariant/testdata'


def diff_fields(a: dict, b: dict):
  return [k for k in a if a[k] != b[k]]


def main():
  golden = [canonical(r) for r in tfrecord.read_records(os.path.join(TESTDATA, 'golden.calling_candidates.tfrecord.gz'))]
  bam_path = os.path.join(TESTDATA, 'input/NA12878_S1.chr20.10_10p1mb.bam')
  ref = fasta.IndexedFastaReader(os.path.join(TESTDATA, 'input/ucsc.hg19.chr20.unittest.fasta.gz'))
  table = bam.NativeBamTable(bam_path, bam.ReadRequirements(min_mapping_quality=5))
  opts = cand.CandidateOptions(sample_name=cand.sample_name_from_bam(bam_path), small_model_vaf_context_window_size=51)
  ours = []
  region = ('chr20', 9999999, 10010000)       # --regions chr20:10,000,000-10,010,000
  for contig, s, e in cand.regions_to_process([(c, ref.n_bases(c)) for c in ref.contig_order], opts.partition_size, region):
    ours += [canonical(r) for r in cand.candidates_in_region(table, ref, contig, s, e, opts).records]
  g_by = {(c['start'], c['ref'], tuple(c['alts'])): c for c in golden}
  o_by = {(c['start'], c['ref'], tuple(c['alts'])): c for c in ours}
  exact, partial, fixture = [], [], []
  for key, g in g_by.items():
    o = o_by.get(key)
    if o is None:
      continue
    d = diff_fields(g, o)
    if not d:
      exact.append(key[0])
      fixture.append(g)
    else:
      partial.append({'start': key[0], 'differs_in': d})
  report = {
      'golden_candidates': len(golden), 'ours_candidates': len(ours), 'sample_name': opts.sample_name,
      'same_site_and_alleles': len(exact) + len(partial), 'identical_in_every_field': len(exact),
      'same_alleles_different_counts_or_support': partial,
      'golden_only': sorted(k[0] for k in g_by if k not in o_by), 'ours_only': sorted(k[0] for k in o_by if k not in g_by),
      'note': 'golden made with --realign_reads (default); ours = no realigner',
  }
  report['pacbio'] = pacbio_pin()
  os.makedirs(os.path.join(ROOT, 'tests/golden'), exist_ok=True)
  with open(os.path.join(ROOT, 'tests/golden/candidates_golden_report.json'), 'w') as f:
    json.dump(report, f, indent=1)
  print(json.dumps({k: v for k, v in report.items() if not isinstance(v, list) or len(v) < 30}, indent=1))
  write_fixture(fixture, g_by, o_by, table, ref, opts)


def pacbio_golden_variants(path: str) -> dict:
  """The variants of golden.pacbio_examples, by (start, ref, alts)."""
  gold = {}
  for r in tfrecord.read_records(path):
    c = canonical(protos.f_bytes(1, protos.parse_tf_example(r)['variant/encoded'][1][0]))
    gold[(c['start'], c['ref'], tuple(c['alts']))] = c
  return gold


def pacbio_pin(bam_path=None, ref_path=None, golden=None, region=('chr20', 8999999, 9100000)):
  """golden.pacbio_examples.tfrecord.gz (make_examples_test.py:792-831: realigner off, --track_ref_reads, --phase_reads region
  padding, --vsc_min_fraction_indels 0.12, --partition_size 25000): every variant/encoded of the 401 examples against ours.
  golden: canonical_call dicts of the golden variants (default: all of golden.pacbio_examples); region: where to call them."""
  if golden is None:
    gold = pacbio_golden_variants(os.path.join(TESTDATA, 'golden.pacbio_examples.tfrecord.gz'))
  else:
    gold = {(c['start'], c['ref'], tuple(c['alts'])): c for c in golden}
  bam_path = bam_path or os.path.join(TESTDATA, 'input/test_pacbio.chr20_100kbp_at_9mb.bam')
  ref = fasta.IndexedFastaReader(ref_path or os.path.join(TESTDATA, 'input/grch38.chr20_and_21_10M.fa.gz'))
  table = bam.NativeBamTable(bam_path, bam.ReadRequirements(min_mapping_quality=1), parse_aux=True)
  opts = cand.CandidateOptions(sample_name=cand.sample_name_from_bam(bam_path), min_mapping_quality=1, track_ref_reads=True,
                               vsc_min_fraction_indels=0.12, partition_size=25000)
  ours = {}
  for contig, s, e in cand.regions_to_process([(c, ref.n_bases(c)) for c in ref.contig_order], 25000, region):
    for rec in cand.candidates_in_region(table, ref, contig, s, e, opts, padding_pct=20).records:
      c = canonical(rec)
      ours[(c['start'], c['ref'], tuple(c['alts']))] = c
  same = [k for k in gold if k in ours and all(gold[k][f] == ours[k][f] for f in ('info', 'call_set_name', 'genotype', 'end', 'contig'))]
  n_examples = sum(1 for _ in tfrecord.read_records(os.path.join(TESTDATA, 'golden.pacbio_examples.tfrecord.gz'))) if golden is None else None
  return {'golden_examples': n_examples, 'golden_variants': len(gold), 'ours_candidates': len(ours),
          'identical_site_alleles_AD_DP_VAF': len(same), 'golden_only': len(set(gold) - set(ours)), 'ours_only': len(set(ours) - set(gold))}


def write_fixture(exact, g_by, o_by, table, ref, opts, n_partitions=3):
  """Portable fixture: the reads (as a small BAM) and reference slice of the partitions whose golden candidates are all
  reproduced field for field, with those golden candidates as the expected output."""
  sys.path.insert(0, os.path.join(ROOT, 'tests'))
  import test_bam_native as tb
  origin, size = 9999999, opts.partition_size
  by_part = {}
  for key, g in g_by.items():
    by_part.setdefault((key[0] - origin) // size, []).append(key)
  ours_by_part = {}
  for key in o_by:
    ours_by_part.setdefault((key[0] - origin) // size, []).append(key)
  good = [p for p, keys in sorted(by_part.items())
          if sorted(keys) == sorted(ours_by_part.get(p, [])) and
          all(diff_fields(g_by[k], o_by[k]) in ([], ['af_at_position']) for k in keys)]
  good = sorted(good, key=lambda p: -len(by_part[p]))[:n_partitions]
  parts, rows_all = [], []
  for p in sorted(good):
    s, e = origin + p * size, origin + (p + 1) * size
    rows = cand.region_reads(table, 'chr20', s, e)
    rows_all += [int(r) for r in rows if int(r) not in rows_all]
    # 'af_exact': the +-25 bp allele-fraction context also matches (it does not where the realigner rewrote a nearby read)
    parts.append({'start': s, 'end': e, 'expected': [dict(g_by[k], af_exact=not diff_fields(g_by[k], o_by[k])) for k in sorted(by_part[p])]})
  rows_all.sort()
  lo = min(int(table.pos[r]) for r in rows_all) - 2
  hi = max(int(table.end[r]) for r in rows_all) + 64
  recs = []
  for r in rows_all:
    rd = table.read(r)
    recs.append(tb._record(0, rd.position, rd.fragment_name, rd.mapping_quality, int(table.flag[r]), rd.cigar,
                           rd.aligned_sequence.decode(), rd.aligned_quality, tlen=rd.fragment_length))
  with open(os.path.join(ROOT, 'tests/golden/candidates_golden_subset.bam'), 'wb') as f:
    f.write(tb._bam(recs, refs=(('chr20', ref.n_bases('chr20')),)))
  with open(os.path.join(ROOT, 'tests/golden/candidates_golden_subset.json'), 'w') as f:
    json.dump({'source': 'deepvariant/testdata/golden.calling_candidates.tfrecord.gz + input/NA12878_S1.chr20.10_10p1mb.bam',
               'contig': 'chr20', 'n_bases': ref.n_bases('chr20'), 'slice_start': lo, 'slice': ref.query('chr20', lo, hi),
               'sample_name': opts.sample_name, 'small_model_vaf_context_window_size': 51, 'partitions': parts}, f)
  print('fixture:', len(rows_all), 'reads,', sum(len(p['expected']) for p in parts), 'golden candidates in partitions', sorted(good))


if __name__ == '__main__':
  main()
