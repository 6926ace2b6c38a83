"""WGS alt-aligned goldens: golden.alt_aligned_pileup_{diff_channels,rows}_examples.tfrecord.gz (deepvariant/make_examples_test.py:739-790,
training mode over chr20:10,000,000-10,010,000 with the realigner; training only drops / labels examples, the images of the examples it
keeps are those of calling mode).  Every golden example is rebuilt from BAM + FASTA: realigner -> candidates -> pileups + alt-aligned
pileups -> diff channels (100 x 221 x 8) or stacked rows (300 x 221 x 6).  Writes tests/golden/alt_aligned_wgs_report.json."""
import hashlib
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


def image_digest(image: bytes, shape) -> str:
  """SHA-256 of an example's image bytes and shape."""
  return hashlib.sha256(bytes(image) + repr([int(x) for x in shape]).encode()).hexdigest()


def run(layout: str, golden_digests=None, bam_path=None, ref_path=None) -> dict:
  """golden_digests: [start, alt allele indices, image_digest] per golden example (default: read from the testdata's goldens)."""
  golden = {}
  if golden_digests is None:
    golden_digests = []
    for r in tfrecord.read_records(T + f'golden.alt_aligned_pileup_{layout}_examples.tfrecord.gz'):
      e = protos.parse_tf_example(r)
      golden_digests.append([protos.parse_variant(e['variant/encoded'][1][0]).start, protos.parse_alt_allele_indices(e['alt_allele_indices/encoded'][1][0]),
                             image_digest(e['image/encoded'][1][0], e['image/shape'][1])])
  for start, idx, digest in golden_digests:
    golden[(start, tuple(idx))] = digest
  ref = fasta.IndexedFastaReader(ref_path or T + 'input/ucsc.hg19.chr20.unittest.fasta.gz')
  table = bam.NativeBamTable(bam_path or T + 'input/NA12878_S1.chr20.10_10p1mb.bam', bam.ReadRequirements(min_mapping_quality=5))
  copts = cand.CandidateOptions(sample_name='NA12878')
  pic = pi.default_options(pi.ReadRequirements(10, 5))
  pic.channels = list(pi.PILEUP_DEFAULT_CHANNELS)
  if layout == 'diff_channels':
    pic.channels += ['diff_channels_alternate_allele_1', 'diff_channels_alternate_allele_2']
  pic.num_channels = len(pic.channels)
  pic.alt_aligned_pileup = layout
  gen = men.ExamplesGenerator(men.MakeExamplesOptions(pic_options=pic), test_mode=True, ref_reader=ref)
  params = pi.to_params(pic)
  rl = realigner.Realigner(ref)
  refs = [(c, ref.n_bases(c)) for c in ref.contig_order]
  stats = dict(layout=layout, golden_examples=len(golden), shape=list(gen.image_shape()), compared=0, images_identical=0,
               examples_with_alt_aligned_pileups=0, of_those_identical=0)
  with tempfile.TemporaryDirectory() as tmp:
    for contig, s, e in cand.regions_to_process(refs, 1000, ('chr20', 9999999, 10010000)):
      rows = cand.region_reads(table, contig, s, e)
      path = os.path.join(tmp, 'r.bam')
      bam.write_bam(path, rl.realign_reads(table, contig, rows, (s, e)), refs)
      t2 = bam.NativeBamTable(path, bam.ReadRequirements(min_mapping_quality=5))
      rows2 = t2.query_indices(contig, s, e)
      found = cand.candidates_in_region(t2, ref, contig, s, e, copts, rows=rows2)
      plans = gen.plan_region(found.calls(), [t2.read(int(i)) for i in rows2], {})
      t2.close()
      if not plans:
        continue
      specs, alt_at = [p.spec for p in plans], []
      for p in plans:
        alt_at.append(list(range(len(specs), len(specs) + len(p.alt_specs))))
        specs += p.alt_specs
      imgs = men.compose_alt_aligned(oracle_lib.encode_batch(params, packing.pack_images(specs, params)), len(plans), alt_at, pic,
                                     [p.alt_combination for p in plans])
      assert list(imgs.shape[1:]) == gen.image_shape()
      for p, img in zip(plans, imgs):
        g = golden.get((p.variant.start, tuple(p.variant.alternate_bases.index(a) for a in p.alt_combination)))
        if g is None:
          continue          # training mode dropped it (outside the confident regions)
        ok = image_digest(np.ascontiguousarray(img).tobytes(), img.shape) == g
        stats['compared'] += 1
        stats['images_identical'] += ok
        if p.alt_specs:
          stats['examples_with_alt_aligned_pileups'] += 1
          stats['of_those_identical'] += ok
  return stats


def main():
  report = [run('diff_channels'), run('rows')]
  with open(os.path.join(ROOT, 'tests/golden/alt_aligned_wgs_report.json'), 'w') as f:
    json.dump(report, f, indent=1)
  print(json.dumps(report, indent=1))


if __name__ == '__main__':
  main()
