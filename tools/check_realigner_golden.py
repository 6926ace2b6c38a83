"""Pins the local realigner (deepvariant_b200/realigner.py + fast_pass_aligner.py + csrc/dvb_ssw.cu) end to end against the reference's
WGS goldens, which were made with --realign_reads (scripts/create_golden.sh:165-176): for every 1-kb partition of
chr20:10,000,000-10,010,000 - region reads -> realigner -> candidates (golden.calling_candidates.tfrecord.gz, 78 DeepVariantCalls,
every field) -> pileups (golden.calling_examples.tfrecord.gz, 84 images of 100 x 221 x 7 through the planner + CPU oracle).
Writes tests/golden/realigner_golden_report.json.

--with_flags pins golden.calling_examples.with_flags.tfrecord.gz instead (scripts/create_golden.sh:472-487: --min_mapping_quality 1
--keep_legacy_allele_counter_behavior --normalize_reads, the VG Giraffe settings): realigner -> deepvariant_b200/normalize_reads.py
-> candidates -> pileups; report in tests/golden/with_flags_golden_report.json (examples only, that golden has no candidates file)."""
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import oracle_lib  # noqa: E402
from deepvariant_b200 import bam, candidates as cand, fasta, packing, protos, realigner, tfrecord  # noqa: E402
from deepvariant_b200 import make_examples_native as men  # noqa: E402
from deepvariant_b200 import pileup_image as pi  # noqa: E402

T = '/root/reference/deepvariant/testdata/'


def decoded_features(e: dict) -> dict:
  """The comparison of assertDeepVariantExamplesEqual (deepvariant/make_examples_test.py:1047-1066): every feature decoded, the two
  serialized protos compared as parsed messages."""
  out = {}
  for k, (kind, vals) in e.items():
    if k == 'variant/encoded':
      c = cand.canonical_call(protos.f_bytes(1, vals[0]))
      out[k] = {f: c[f] for f in ('ref', 'alts', 'start', 'end', 'contig', 'info', 'call_set_name', 'genotype')}
    elif k == 'alt_allele_indices/encoded':
      out[k] = protos.parse_alt_allele_indices(vals[0])
    elif kind == 'bytes':
      out[k] = [bytes(v) for v in vals]
    else:
      out[k] = list(vals)
  return out


def main(with_flags=False, td=T, bam_path=None, ref_path=None, shard_keys=None, write=True):
  """Compares with the goldens in the testdata directory td; bam_path / ref_path default to its inputs, shard_keys (the
  [start, alt allele indices] of each --task shard's examples) to its three shard files.  Returns the report."""
  from deepvariant_b200 import normalize_reads
  min_mapq = 1 if with_flags else 5
  examples_golden = 'golden.calling_examples.with_flags.tfrecord.gz' if with_flags else 'golden.calling_examples.tfrecord.gz'
  golden_c = [] if with_flags else [cand.canonical_call(r) for r in tfrecord.read_records(os.path.join(td, 'golden.calling_candidates.tfrecord.gz'))]
  golden_e, golden_features, golden_order = {}, {}, []
  for r in tfrecord.read_records(os.path.join(td, examples_golden)):
    e = protos.parse_tf_example(r)
    v = protos.parse_variant(e['variant/encoded'][1][0])
    idx = tuple(protos.parse_alt_allele_indices(e['alt_allele_indices/encoded'][1][0]))
    golden_e[(v.start, idx)] = np.frombuffer(e['image/encoded'][1][0], dtype=np.uint8).reshape(e['image/shape'][1])
    golden_features[(v.start, idx)] = decoded_features(e)
    golden_order.append((v.start, idx))
  golden_shards = []
  for i in range(0 if with_flags else 3):
    keys = []
    if shard_keys is not None:
      keys = [(k[0], tuple(k[1])) for k in shard_keys[i]]
    else:
      for r in tfrecord.read_records(os.path.join(td, f'golden.calling_examples.tfrecord.gz-0000{i}-of-00003')):
        e = protos.parse_tf_example(r)
        keys.append((protos.parse_variant(e['variant/encoded'][1][0]).start, tuple(protos.parse_alt_allele_indices(e['alt_allele_indices/encoded'][1][0]))))
    golden_shards.append(keys)
  bam_path = bam_path or os.path.join(td, 'input/NA12878_S1.chr20.10_10p1mb.bam')
  ref = fasta.IndexedFastaReader(ref_path or os.path.join(td, 'input/ucsc.hg19.chr20.unittest.fasta.gz'))
  table = bam.NativeBamTable(bam_path, bam.ReadRequirements(min_mapping_quality=min_mapq))
  copts = cand.CandidateOptions(sample_name=cand.sample_name_from_bam(bam_path), small_model_vaf_context_window_size=51,
                                min_mapping_quality=min_mapq, keep_legacy_allele_counter_behavior=with_flags)
  pic = pi.default_options(pi.ReadRequirements(min_base_quality=10, min_mapping_quality=min_mapq))
  pic.channels = list(pi.PILEUP_CHANNELS_WITH_INSERT_SIZE)
  pic.num_channels = 7
  gen = men.ExamplesGenerator(men.MakeExamplesOptions(pic_options=pic), test_mode=True, ref_reader=ref)
  params = pi.to_params(pic)
  ropts = realigner.RealignerOptions(normalize_reads=with_flags)
  ropts.ws.keep_legacy_behavior = with_flags                  # realigner.py:345-360, 414-429 take both flags over
  rl = realigner.Realigner(ref, ropts)
  refs = [(c, ref.n_bases(c)) for c in ref.contig_order]
  ours_c, images, n_windows = [], {}, 0
  n_normalized = n_heading = 0
  ours_features, ours_order, region_keys = {}, [], []
  with tempfile.TemporaryDirectory() as tmp:
    for contig, s, e in cand.regions_to_process(refs, 1000, ('chr20', 9999999, 10010000)):
      rows = cand.region_reads(table, contig, s, e)
      reads = rl.realign_reads(table, contig, rows, (s, e))
      count_reads = None
      if with_flags:
        before = reads
        reads, count_reads = normalize_reads.normalize_region_reads(reads, lambda a, b: ref.query(contig, a, b).encode(), s, e, ref.n_bases(contig), min_mapq)
        n_normalized += sum(1 for a, b in zip(reads, before) if a is not b)
      t2 = bam.scratch_table(reads, refs, bam.ReadRequirements(min_mapping_quality=min_mapq))
      assert t2.n_reads == len(reads), (t2.n_reads, len(reads))
      rows2 = t2.query_indices(contig, s, e)
      if count_reads is None:
        found = cand.candidates_in_region(t2, ref, contig, s, e, copts, rows=rows2)
      else:            # reads whose only change is the heading indel are counted with it, piled up without it
        n_heading += 1
        tc = bam.scratch_table(count_reads, refs, bam.ReadRequirements(min_mapping_quality=min_mapq))
        found = cand.candidates_in_region(tc, ref, contig, s, e, copts, rows=tc.query_indices(contig, s, e))
        tc.close()
      ours_c += [cand.canonical_call(r) for r in found.records]
      plans = gen.plan_region(found.calls(), [t2.read(int(i)) for i in rows2], {})
      if plans:
        imgs = oracle_lib.encode_batch(params, packing.pack_images([p.spec for p in plans], params))
        keys = []
        for p, img in zip(plans, imgs):
          key = (p.variant.start, tuple(p.variant.alternate_bases.index(a) for a in p.alt_combination))
          images[key] = img
          ours_features[key] = decoded_features(protos.parse_tf_example(gen.encode_example(p, img, {})))
          ours_order.append(key)
          keys.append(key)
        region_keys.append(keys)
      else:
        region_keys.append([])
      t2.close()
  g_by = {(c['start'], c['ref'], tuple(c['alts'])): c for c in golden_c}
  o_by = {(c['start'], c['ref'], tuple(c['alts'])): c for c in ours_c}
  both = [k for k in g_by if k in o_by]
  exact = [k for k in both if g_by[k] == o_by[k]]
  partial = [{'start': k[0], 'differs_in': [f for f in g_by[k] if g_by[k][f] != o_by[k][f]]} for k in both if g_by[k] != o_by[k]]
  img_eq = [k for k in golden_e if k in images and np.array_equal(images[k], golden_e[k])]
  rows_total = rows_hit = 0
  for k, g in golden_e.items():
    if k in images:
      g_rows = [g[r].tobytes() for r in range(5, 100) if g[r].any()]
      o_rows = set(images[k][r].tobytes() for r in range(5, 100) if images[k][r].any())
      rows_total += len(g_rows)
      rows_hit += sum(1 for r in g_rows if r in o_rows)
  # --task i of 3: region j goes to task j mod 3 (regions_to_process), records in region order within a shard
  shards_equal = [sum((region_keys[j] for j in range(i, len(region_keys), 3)), []) == golden_shards[i] for i in range(len(golden_shards))]
  features_equal = sum(1 for k in golden_features if ours_features.get(k) == golden_features[k])
  report = {'with_flags': with_flags, 'reads_rewritten_by_normalization': n_normalized, 'regions_with_heading_indel_only_reads': n_heading, 'tf_examples_equal_feature_by_feature': features_equal, 'example_order_equal': ours_order == golden_order,
            'sharded_goldens_equal_task_by_task': shards_equal, 'golden_candidates': len(golden_c), 'ours_candidates': len(ours_c), 'same_site_and_alleles': len(both),
            'candidates_identical_in_every_field': len(exact), 'candidates_partial': partial,
            'golden_only': sorted(k[0] for k in g_by if k not in o_by), 'ours_only': sorted(k[0] for k in o_by if k not in g_by),
            'golden_examples': len(golden_e), 'examples_planned': len(images), 'images_identical': len(img_eq),
            'golden_read_rows': rows_total, 'golden_read_rows_reproduced': rows_hit}
  if write:
    with open(os.path.join(ROOT, 'tests/golden/' + ('with_flags_golden_report.json' if with_flags else 'realigner_golden_report.json')), 'w') as f:
      json.dump(report, f, indent=1)
    print(json.dumps({k: v for k, v in report.items() if not isinstance(v, list) or len(v) < 20}, indent=1))
    for p in partial[:10]:
      print(p)
  return report


if __name__ == '__main__':
  main('--with_flags' in sys.argv[1:])
