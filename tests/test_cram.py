"""CRAM 3.0 input (csrc/dvb_cram.cu -> dvb_cram_to_bam): the reference's own small CRAM vectors (tests/golden/cram/, copied by
tools/make_cram_fixtures.py) against the SAM they were written from, and the first container of the reference's chr20 CRAM against
its BAM, read for read (make_examples_test.py:330-372 expects the BAM's goldens from that CRAM)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepvariant_b200 import _lib, bam, candidates as cand, fasta  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
CRAM = os.path.join(GOLDEN, 'cram')
# The reference's chr20 CRAM cut to its first container (10,000 records from chr20:9,999,912), the records of its BAM that start
# before chr20:10,011,000, and the reference bases of chr20:9,990,000-10,020,000 (tools/make_reference_subset_fixtures.py).
CHR20_CRAM = os.path.join(GOLDEN, 'NA12878_S1.chr20.10_10p1mb.first_container.cram')
CHR20_BAM = os.path.join(GOLDEN, 'NA12878_S1.chr20.10_10p1mb.window.bam')
CHR20_FASTA = os.path.join(GOLDEN, 'quickstart.chr20_10mb.fa.gz')


def _keep_all():
  req = bam.ReadRequirements(min_mapping_quality=0)
  req.keep_duplicates = req.keep_failed_vendor_quality_checks = req.keep_secondary_alignments = req.keep_supplementary_alignments = True
  req.keep_unaligned = req.keep_improperly_placed = True
  return req


def _sam_records(path):
  out = []
  for line in open(path):
    if line.startswith('@'):
      continue
    t = line.rstrip('\n').split('\t')
    out.append(dict(name=t[0], flag=int(t[1]), contig=t[2], pos=int(t[3]) - 1, mapq=int(t[4]), cigar=t[5], mate_pos=int(t[7]) - 1, tlen=int(t[8]),
                    seq=t[9], qual=bytes(ord(c) - 33 for c in t[10]), tags={x[:2]: x[5:] for x in t[11:]}))
  return out


def _cigar_text(read):
  return ''.join(f'{n}{"MIDNSHP=X"[op]}' for op, n in read.cigar)


@pytest.mark.parametrize('embedded', [0, 1])
def test_small_cram_vectors_equal_their_sam(embedded, tmp_path):
  ref = fasta.IndexedFastaReader(os.path.join(CRAM, 'test.fasta'))
  path = os.path.join(CRAM, f'test_cram.embed_ref_{embedded}_version_3.0.cram')
  assert bam.is_cram(path) and not bam.is_cram(os.path.join(CRAM, 'test.fasta'))
  table = bam.NativeBamTable(path, _keep_all(), parse_aux=True, ref_reader=ref)
  want = _sam_records(os.path.join(CRAM, 'test_cram.sam'))
  assert table.n_reads == len(want) == 3 and table.references == ['chrM', 'chr1', 'chr2'] and table.reference_lengths == [100, 76, 121]
  for i, w in enumerate(want):
    r = table.read(i)
    assert (r.fragment_name, r.reference_name, r.position, r.mapping_quality, _cigar_text(r)) == (w['name'], w['contig'], w['pos'], w['mapq'], w['cigar'])
    assert r.aligned_sequence.decode() == w['seq'] and bytes(r.aligned_quality) == w['qual']
    assert int(table.flag[i]) == w['flag'] and int(table.fragment_length[i]) == w['tlen']
  # the records' aux fields come back BAM-encoded: integer tags with the values of the SAM
  aux = table.aux[int(table.aux_begin[2]):int(table.aux_begin[3])]
  k = aux.index(b'ZA')
  assert aux[k + 2:k + 3] in (b's', b'S') and int.from_bytes(aux[k + 3:k + 5], 'little') == 275          # ZA:i:275 of the SAM
  assert 'SM' not in bam.sam_header_text(path) and bam.sam_header_text(path).startswith('@HD')
  assert cand.sample_name_from_bam(path) == cand.DEFAULT_SAMPLE_NAME
  if embedded:
    # the slice carries its own reference: no FASTA contig is needed
    class NoContigs:
      contig_order = []
    assert bam.NativeBamTable(path, _keep_all(), ref_reader=NoContigs()).n_reads == 3
  else:
    class NoContigs:
      contig_order = []
    with pytest.raises(_lib.DvbError, match='reference bases of chr1 are needed'):
      bam.NativeBamTable(path, _keep_all(), ref_reader=NoContigs())
  with pytest.raises(ValueError, match='reference FASTA is needed'):
    bam.NativeBamTable(path, _keep_all())
  # regions: containers that do not overlap are skipped, the BAM reader filters the rest
  assert bam.NativeBamTable(path, _keep_all(), ref_reader=ref, regions=[('chr1', 50, 60)]).n_reads == 3
  assert bam.NativeBamTable(path, _keep_all(), ref_reader=ref, regions=[('chr1', 70, 76)]).n_reads == 1          # only the 41M read reaches 70
  assert bam.NativeBamTable(path, _keep_all(), ref_reader=ref, regions=[('chr2', 0, 100)]).n_reads == 0
  assert bam.NativeBamTable(path, _keep_all(), ref_reader=ref, regions=[('chrM', 0, 100)]).n_reads == 0


def test_cram_argument_errors(tmp_path):
  lib = _lib.lib()
  junk = tmp_path / 'junk.cram'
  junk.write_bytes(b'CRAM\x03\x00' + b'\0' * 20 + b'\x10\x00\x00\x00' + b'\xff' * 40)
  with pytest.raises(_lib.DvbError):
    _lib.check(lib.dvb_cram_to_bam(str(junk).encode(), str(tmp_path / 'o.bam').encode(), None, None, None, 0, None, None, None, 0, None))
  v2 = tmp_path / 'v2.cram'
  v2.write_bytes(b'CRAM\x02\x01' + b'\0' * 40)
  with pytest.raises(_lib.DvbError, match='CRAM 2.1'):
    _lib.check(lib.dvb_cram_to_bam(str(v2).encode(), str(tmp_path / 'o.bam').encode(), None, None, None, 0, None, None, None, 0, None))
  with pytest.raises(_lib.DvbError, match='not a CRAM'):
    _lib.check(lib.dvb_cram_to_bam(os.path.join(CRAM, 'test.fasta').encode(), str(tmp_path / 'o.bam').encode(), None, None, None, 0, None, None, None, 0, None))
  with pytest.raises(_lib.DvbError):
    _lib.check(lib.dvb_cram_to_bam(None, None, None, None, None, 0, None, None, None, 0, None))
  # a truncated copy of a good file: an error, never a crash
  good = open(os.path.join(CRAM, 'test_cram.embed_ref_1_version_3.0.cram'), 'rb').read()
  for cut in (30, 200, 900, len(good) - 60):
    p = tmp_path / f'cut{cut}.cram'
    p.write_bytes(good[:cut])
    rc = lib.dvb_cram_to_bam(str(p).encode(), str(tmp_path / 'o.bam').encode(), None, None, None, 0, None, None, None, 0, None)
    assert rc in (0, 1, 7)


def test_reference_chr20_cram_equals_its_bam_read_for_read():
  """The reads of the CRAM's first container that start before chr20:10,010,000 against the same reads of the BAM: gzip and rANS
  (order 0 and 1) blocks, mates linked inside the slices and detached ones, every field the table holds."""
  ref = fasta.IndexedFastaReader(CHR20_FASTA)
  assert bam.NativeBamTable(CHR20_CRAM, _keep_all(), ref_reader=ref).n_reads == 10000
  whole = [('chr20', 0, 10_010_000)]       # every read of the BAM fixture starting before 10,010,000, and no read past the container
  c = bam.NativeBamTable(CHR20_CRAM, _keep_all(), parse_aux=True, ref_reader=ref, regions=whole)
  b = bam.NativeBamTable(CHR20_BAM, _keep_all(), parse_aux=True, regions=whole)
  assert c.n_reads == b.n_reads == 4986
  for name in ('ref_id', 'pos', 'end', 'mapq', 'flag', 'fragment_length', 'hp', 'read_number', 'number_reads', 'seq_begin', 'cigar_begin', 'name_begin',
               'bases', 'quals', 'cigar'):
    np.testing.assert_array_equal(getattr(c, name), getattr(b, name), err_msg=name)
  assert c.names == b.names
  # a region-restricted open gives the rows the BAM's region open gives
  regions = [('chr20', 10005000, 10006000)]
  cr = bam.NativeBamTable(CHR20_CRAM, _keep_all(), ref_reader=ref, regions=regions)
  br = bam.NativeBamTable(CHR20_BAM, _keep_all(), regions=regions)
  assert cr.n_reads == br.n_reads > 100 and cr.reads() == br.reads()
  assert cand.sample_name_from_bam(CHR20_CRAM) == 'NA12878'


def test_make_examples_over_the_cram_writes_the_goldens_of_the_bam(tmp_path, monkeypatch):
  """make_examples_test.py:330-372 (TestConditions.USE_CRAM): --reads NA12878_S1.chr20.10_10p1mb.cram must give golden.calling_examples.
  The encoder is the CPU oracle here; reads, realigner, candidates and planning are the product flow."""
  sys.path.insert(0, os.path.join(ROOT, 'tests'))
  import test_candidates as tc
  from deepvariant_b200 import cli, make_examples_native as men, pileup_image as pi, protos, tfrecord
  monkeypatch.setattr(men.ExamplesGenerator, '_gpu', lambda self: tc.OracleEncoder(pi.to_params(self.options.pic_options, height=self.pileup_image_height)))
  out = str(tmp_path / 'examples.tfrecord.gz')
  assert cli.make_examples(['--mode', 'calling', '--ref', CHR20_FASTA,
                            '--reads', CHR20_CRAM, '--regions', 'chr20:10,000,000-10,010,000',
                            '--examples', out, '--channel_list', 'BASE_CHANNELS,insert_size']) == 0
  golden = [protos.parse_tf_example(r) for r in tfrecord.read_records(os.path.join(GOLDEN, 'golden.calling_examples.tfrecord.gz'))]
  ours = [protos.parse_tf_example(r) for r in tfrecord.read_records(out)]
  assert len(ours) == len(golden) == 84
  for g, o in zip(golden, ours):
    for key in ('image/encoded', 'image/shape', 'alt_allele_indices/encoded', 'locus'):
      assert g[key] == o[key], key
