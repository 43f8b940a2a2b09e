"""Record-path parity (CPU): TFRecord framing / CRC-32C / tf.Example parsing / image decode of the
host side of libt2r_b200.so against the pure-Python oracle and the golden values of the reference's
own fixture test_data/pose_env_test_data.tfrecord (tests/golden/pose_env_golden.npz).

Mirrors the assertions of the reference's utils/tfdata_test.py: fixture shapes (:65-88), PNG
uint8/uint16 (:143-179), unsupported dtype raises (:181-202), varlen ints (:230-248), wrong image
size raises (:311-344), file-pattern inference (:398-433), get_batch_size (:436-444).
"""
import ctypes as C
import io
import os

import numpy as np
import pytest
from PIL import Image

from oracle import tfrecord as oracle
from tensor2robot_b200 import _lib
from tensor2robot_b200.utils import dtypes
from tensor2robot_b200.utils import tensorspec_utils as utils
from tensor2robot_b200.utils import tfdata

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, 'golden', 'pose_env_test_data.tfrecord')
GOLDEN = np.load(os.path.join(HERE, 'golden', 'pose_env_golden.npz'))
TSPEC = utils.ExtendedTensorSpec


@pytest.fixture(autouse=True)
def _host_image_decoder(monkeypatch):
  """The host decoder (numpy out) on every machine: 'auto' picks the device decoder where a GPU is present, and
  tests/test_jpeg.py checks that one against this one."""
  monkeypatch.setattr(tfdata, 'IMAGE_DECODER', 'host')


def test_library_exports_every_declared_symbol():
  lib = _lib.lib()
  header = open(os.path.join(os.path.dirname(HERE), 'include', 't2r_b200.h')).read()
  import re
  declared = set(re.findall(r'\b(t2r_[a-z0-9_]+)\s*\(', header))
  assert declared, 'no declarations found'
  for name in sorted(declared):
    assert hasattr(lib, name), name
  assert set(_lib.EXPORTED_SYMBOLS) <= declared | {'t2r_version'}
  assert lib.t2r_version() >= 100


def test_crc32c_known_answers():
  lib = _lib.lib()
  vectors = [(b'', 0x00000000), (b'a', 0xC1D04330), (b'123456789', 0xE3069283), (bytes(32), 0x8A9136AA),
             (bytes([0xFF] * 32), 0x62A8AB43), (bytes(range(32)), 0x46DD794E)]   # RFC 3720 B.4 vectors
  for data, expected in vectors:
    buf = C.create_string_buffer(data, len(data))
    assert lib.t2r_crc32c(C.addressof(buf), len(data)) == expected, data
    assert oracle.crc32c(data) == expected
    assert lib.t2r_masked_crc32c(C.addressof(buf), len(data)) == oracle.masked_crc32c(data)
  try:
    from tensorboard.compat.tensorflow_stub.pywrap_tensorflow import masked_crc32c
  except Exception:  # pragma: no cover
    return
  rng = np.random.RandomState(0)
  for n in (1, 7, 8, 9, 63, 64, 1000):
    data = rng.bytes(n)
    buf = C.create_string_buffer(data, n)
    assert lib.t2r_masked_crc32c(C.addressof(buf), n) == masked_crc32c(data)


def test_fixture_framing_matches_oracle():
  f = tfdata.TFRecordFile(FIXTURE, verify_crc=True)
  ref = oracle.read_tfrecords(FIXTURE)
  assert len(f) == len(ref) == 100
  np.testing.assert_array_equal(f.lengths, GOLDEN['record_length'])
  assert list(f) == ref


def test_corrupt_record_is_rejected(tmp_path):
  data = bytearray(open(FIXTURE, 'rb').read())
  data[40] ^= 0x01
  bad = tmp_path / 'bad.tfrecord'
  bad.write_bytes(bytes(data))
  with pytest.raises(ValueError):
    tfdata.TFRecordFile(str(bad), verify_crc=True)
  assert len(tfdata.TFRecordFile(str(bad), verify_crc=False)) == 100
  bad.write_bytes(bytes(data[:-3]))
  with pytest.raises(ValueError):
    tfdata.TFRecordFile(str(bad), verify_crc=False)


def _pose_env_specs():
  features = utils.TensorSpecStruct(
      state=utils.TensorSpecStruct(image=TSPEC((64, 64, 3), dtypes.uint8, 'state/image', data_format='jpeg')),
      action=utils.TensorSpecStruct(pose=TSPEC((2,), dtypes.float32, 'pose')))
  labels = utils.TensorSpecStruct(reward=TSPEC((1,), dtypes.float32, 'reward'),
                                  target_pose=TSPEC((2,), dtypes.float32, 'target_pose'))
  return features, labels


def test_fixture_parses_bit_exact():
  feature_spec, label_spec = _pose_env_specs()
  records = tfdata.read_records(FIXTURE)
  parse = tfdata.create_parse_tf_example_fn(feature_spec, label_spec)
  features, labels = parse(records)
  assert features.state.image.shape == (100, 64, 64, 3) and features.state.image.dtype == np.uint8
  np.testing.assert_array_equal(features.action.pose.view(np.uint32), GOLDEN['pose'].view(np.uint32))
  np.testing.assert_array_equal(labels.reward.view(np.uint32), GOLDEN['reward'].view(np.uint32))
  np.testing.assert_array_equal(labels.target_pose.view(np.uint32), GOLDEN['target_pose'].view(np.uint32))
  np.testing.assert_array_equal(features.state.image.astype(np.int64).sum((1, 2, 3)), GOLDEN['image_sum'])
  np.testing.assert_array_equal(features.state.image[:, :2, :2], GOLDEN['image_corner'])
  # the oracle parser agrees record by record
  for i in (0, 17, 99):
    ex = oracle.parse_example(records[i])
    np.testing.assert_array_equal(np.float32(ex['pose'][1]), features.action.pose[i])
  # zero-copy pointers from the mmap index give the same result
  f = tfdata.TFRecordFile(FIXTURE)
  f2, _ = parse([f.pointer(i) for i in range(5)])
  np.testing.assert_array_equal(f2.action.pose, features.action.pose[:5])


def _png(arr):
  buf = io.BytesIO()
  Image.fromarray(arr.squeeze() if arr.shape[-1] == 1 else arr).save(buf, format='PNG')
  return buf.getvalue()


def test_png_uint8_uint16_and_unsupported_dtype():
  rng = np.random.RandomState(1)
  img8 = rng.randint(0, 255, (12, 10, 1)).astype(np.uint8)
  img16 = rng.randint(0, 65535, (12, 10, 1)).astype(np.uint16)
  rec = oracle.make_example({'a': _png(img8), 'b': _png(img16)})
  spec = utils.TensorSpecStruct(a=TSPEC((12, 10, 1), dtypes.uint8, 'a', data_format='png'),
                                b=TSPEC((12, 10, 1), dtypes.uint16, 'b', data_format='png'))
  out = tfdata.create_parse_tf_example_fn(spec)([rec, rec])
  np.testing.assert_array_equal(out.a[1], img8)
  np.testing.assert_array_equal(out.b[0], img16)
  bad = utils.TensorSpecStruct(a=TSPEC((12, 10, 1), dtypes.uint32, 'a', data_format='png'))
  with pytest.raises(ValueError):
    tfdata.create_parse_tf_example_fn(bad)([rec])


def test_varlen_optional_missing_and_wrong_size():
  rec1 = oracle.make_example({'ids': [1, 2], 'x': [0.5, 1.5, 2.5]})
  rec2 = oracle.make_example({'ids': [1, 2, 3, 4, 5], 'x': [1.0, 2.0, 3.0]})
  spec = utils.TensorSpecStruct(ids=TSPEC((3,), dtypes.int64, 'ids', varlen_default_value=3.0),
                                x=TSPEC((3,), dtypes.float32, 'x'),
                                opt=TSPEC((2,), dtypes.float32, 'opt', is_optional=True))
  out = tfdata.create_parse_tf_example_fn(spec)([rec1, rec2])
  np.testing.assert_array_equal(out.ids, [[1, 2, 3], [1, 2, 3]])       # padded with 3, clipped to 3
  np.testing.assert_array_equal(out.x, [[0.5, 1.5, 2.5], [1, 2, 3]])
  with pytest.raises(ValueError):                                        # required key missing
    tfdata.create_parse_tf_example_fn(utils.TensorSpecStruct(y=TSPEC((1,), dtypes.float32, 'y')))([rec1])
  with pytest.raises(ValueError):                                        # wrong number of values
    tfdata.create_parse_tf_example_fn(utils.TensorSpecStruct(x=TSPEC((2,), dtypes.float32, 'x')))([rec1])
  img = np.zeros((8, 8, 3), np.uint8)
  buf = io.BytesIO()
  Image.fromarray(img).save(buf, format='JPEG')
  rec = oracle.make_example({'im': buf.getvalue()})
  with pytest.raises(ValueError):                                        # decoded size != spec
    tfdata.create_parse_tf_example_fn(utils.TensorSpecStruct(
        im=TSPEC((8, 9, 3), dtypes.uint8, 'im', data_format='jpeg')))([rec])
  empty = oracle.make_example({'im': b''})
  out = tfdata.create_parse_tf_example_fn(utils.TensorSpecStruct(
      im=TSPEC((8, 8, 3), dtypes.uint8, 'im', data_format='jpeg')))([empty])
  assert out.im.shape == (1, 8, 8, 3) and not out.im.any()               # '' -> black image


def test_same_name_feeds_several_paths_and_dataset_keys():
  rec_a = oracle.make_example({'v': [1.0]})
  rec_b = oracle.make_example({'v': [2.0]})
  spec = utils.TensorSpecStruct(first=TSPEC((1,), dtypes.float32, 'v', dataset_key='a'),
                                second=TSPEC((1,), dtypes.float32, 'v', dataset_key='b'),
                                third=TSPEC((1,), dtypes.float32, 'v', dataset_key='a'))
  out = tfdata.create_parse_tf_example_fn(spec)({'a': [rec_a], 'b': [rec_b]})
  assert out.first[0, 0] == 1.0 and out.second[0, 0] == 2.0 and out.third[0, 0] == 1.0


def test_file_patterns_and_batch_size(tmp_path):
  assert tfdata.infer_data_format('a/b.tfrecord') == 'tfrecord'
  with pytest.raises(ValueError):
    tfdata.infer_data_format('a/b.tfrecord,c.recordio')
  with pytest.raises(ValueError):
    tfdata.infer_data_format('a/b.txt')
  p = tmp_path / 'x.tfrecord'
  oracle.write_tfrecords(str(p), [oracle.make_example({'v': [float(i)]}) for i in range(10)])
  fmt, files = tfdata.get_data_format_and_filenames('tfrecord:%s,%s' % (p, FIXTURE))
  assert fmt == 'tfrecord' and files == [str(p), FIXTURE]
  with pytest.raises(ValueError):
    tfdata.get_data_format_and_filenames(str(tmp_path / 'missing*.tfrecord'))
  assert tfdata.get_batch_size({'batch_size': 4}, 8) == 4 and tfdata.get_batch_size({}, 8) == 8
  with pytest.raises(ValueError):
    tfdata.get_batch_size({}, None)
  # written records round-trip through the C++ reader
  assert [oracle.parse_example(r)['v'][1][0] for r in tfdata.read_records(str(p))] == [float(i) for i in range(10)]


def test_record_input_generator_batches_and_shards():
  from tensor2robot_b200.input_generators import default_input_generator as gens
  feature_spec, label_spec = _pose_env_specs()
  g = gens.DefaultRecordInputGenerator(file_patterns=FIXTURE, batch_size=32, seed=0)
  g.set_feature_specifications(feature_spec, feature_spec)
  g.set_label_specifications(label_spec, label_spec)
  batches = list(g.create_dataset('eval'))
  assert len(batches) == 3                                   # 100 records, drop_remainder
  f, l = batches[0]
  assert f.state.image.shape == (32, 64, 64, 3) and l.reward.shape == (32, 1)
  np.testing.assert_array_equal(f.action.pose, GOLDEN['pose'][:32])     # eval: file order
  it = g.create_dataset('train')                             # train: shuffled, repeats forever
  seen = [next(it)[0].action.pose for _ in range(5)]
  assert not np.array_equal(seen[0], GOLDEN['pose'][:32])
  # rank sharding by record when there are fewer files than ranks
  g0 = gens.DefaultRecordInputGenerator(file_patterns=FIXTURE, batch_size=10, shard=(0, 2))
  g1 = gens.DefaultRecordInputGenerator(file_patterns=FIXTURE, batch_size=10, shard=(1, 2))
  for g_ in (g0, g1):
    g_.set_feature_specifications(feature_spec, feature_spec)
    g_.set_label_specifications(label_spec, label_spec)
  a = np.concatenate([b[0].action.pose for b in g0.create_dataset('eval')])
  b = np.concatenate([b[0].action.pose for b in g1.create_dataset('eval')])
  np.testing.assert_array_equal(a, GOLDEN['pose'][0::2])
  np.testing.assert_array_equal(b, GOLDEN['pose'][1::2])
  rnd = gens.DefaultRandomInputGenerator(batch_size=3)
  rnd.set_feature_specifications(feature_spec, feature_spec)
  rnd.set_label_specifications(label_spec, label_spec)
  f, l = next(rnd.create_dataset('train'))
  assert f.state.image.shape == (3, 64, 64, 3) and f.state.image.dtype == np.uint8


def test_sequence_example_parsing():
  """utils/tfdata_test.py:346-395 (test_sequence_parsing): image + float sequences from
  feature_lists, an int64 context feature, `<key>_length` outputs, zero padding to the longest
  sequence of the batch (tf.io.parse_sequence_example)."""
  base = (np.arange(8 * 8 * 3).reshape(8, 8, 3) % 7 * 30).astype(np.uint8)

  def record(n_steps):
    imgs, acts = [], []
    for i in range(n_steps):
      buf = io.BytesIO()
      Image.fromarray((base * i % 251).astype(np.uint8)).save(buf, format='PNG')
      imgs.append(buf.getvalue())
      acts.append([3.0, 1.0 + i])
    return oracle.make_sequence_example({'context_feature': [10]},
                                        {'sequence_feature': acts, 'image_sequence_feature': imgs})

  feature_tspec = utils.TensorSpecStruct(
      state=TSPEC((8, 8, 3), dtypes.uint8, 'image_sequence_feature', is_sequence=True, data_format='png'),
      action=TSPEC((2,), dtypes.float32, 'sequence_feature', is_sequence=True))
  feature_tspec = utils.add_sequence_length_specs(feature_tspec)
  label_tspec = utils.add_sequence_length_specs(
      utils.TensorSpecStruct(reward=TSPEC((), dtypes.int64, 'context_feature')))
  parse = tfdata.create_parse_tf_example_fn(feature_tspec, label_tspec)
  for batch in ([record(3)], [record(3), record(3)], [record(3), record(1)]):
    features, labels = parse(batch)
    b = len(batch)
    assert features.state.shape == (b, 3, 8, 8, 3) and features.state.dtype == np.uint8
    assert features.action.shape == (b, 3, 2)
    assert labels.reward.shape == (b,) and labels.reward.tolist() == [10] * b
    for i in range(3):
      np.testing.assert_array_equal(features.state[0, i], (base * i % 251).astype(np.uint8))
      np.testing.assert_array_equal(features.action[0, i], [3.0, 1.0 + i])
  assert features.state_length.tolist() == [3, 1] and features.action_length.tolist() == [3, 1]
  assert not features.state[1, 1:].any() and not features.action[1, 1:].any()   # padding
  # a record without the feature list is a zero-length sequence (allow_missing=True)
  features, _ = parse([oracle.make_sequence_example({'context_feature': [10]}, {})])
  assert features.action.shape == (1, 0, 2) and features.action_length.tolist() == [0]


def test_example_parser_property_round_trip():
  """Property test (hypothesis): random feature dictionaries serialised by the oracle's wire-format writer
  come back bit-exactly through the C++ parser, for float / int64 / bytes features of random shapes."""
  import hypothesis
  from hypothesis import strategies as st

  floats = st.lists(st.floats(width=32, allow_nan=False, allow_infinity=False), min_size=1, max_size=6)
  ints = st.lists(st.integers(min_value=-2**62, max_value=2**62), min_size=1, max_size=6)
  blobs = st.binary(min_size=0, max_size=40)

  @hypothesis.settings(max_examples=60, deadline=None)
  @hypothesis.given(st.lists(st.tuples(floats, ints, blobs), min_size=1, max_size=4))
  def check(rows):
    n_f, n_i = len(rows[0][0]), len(rows[0][1])
    rows = [r for r in rows if len(r[0]) == n_f and len(r[1]) == n_i] or rows[:1]
    spec = utils.TensorSpecStruct(f=TSPEC((n_f,), dtypes.float32, 'f'), i=TSPEC((n_i,), dtypes.int64, 'i'),
                                  s=TSPEC((), dtypes.string, 's'))
    records = [oracle.make_example({'f': r[0], 'i': [int(v) for v in r[1]], 's': r[2]}) for r in rows]
    out = tfdata.create_parse_tf_example_fn(spec)(records)
    np.testing.assert_array_equal(out.f, np.array([r[0] for r in rows], np.float32))
    np.testing.assert_array_equal(out.i, np.array([r[1] for r in rows], np.int64))
    assert [bytes(x) for x in out.s] == [r[2] for r in rows]
    for rec in records:                      # and the oracle reader agrees with its own writer
      back = oracle.parse_example(rec)
      assert back['s'][1] == [rows[records.index(rec)][2]] or back['s'][1] == []

  check()


def test_prefetcher_order_errors_and_shutdown():
  """train_eval.Prefetcher: same items in the same order, producer exceptions surface in the consumer,
  an abandoned iterator stops its thread."""
  import threading
  import time
  from tensor2robot_b200.utils import train_eval
  assert list(train_eval.Prefetcher(iter(range(50)), depth=3)) == list(range(50))
  assert list(train_eval.Prefetcher(iter([]), depth=1)) == []

  def boom():
    yield 1
    yield 2
    raise KeyError('bad record')

  it = train_eval.Prefetcher(boom(), depth=2)
  assert next(it) == 1 and next(it) == 2
  with pytest.raises(KeyError):
    next(it)
  with pytest.raises(KeyError):      # stays failed
    next(it)

  produced = []

  def endless():
    i = 0
    while True:
      produced.append(i)
      yield i
      i += 1

  it = train_eval.Prefetcher(endless(), depth=2)
  assert next(it) == 0
  before = threading.active_count()
  it.close()
  time.sleep(0.5)
  n = len(produced)
  time.sleep(0.3)
  assert len(produced) == n and threading.active_count() <= before    # producer stopped


def test_dataset_metadata_parallel_read_and_parsed_stream(tmp_path):
  """utils/tfdata.py:143-238: shard statistics, interleaved shard reading, parsing an iterable of serialized batches."""
  from oracle import tfrecord
  records = tfrecord.read_tfrecords(FIXTURE)
  for shard in range(3):
    tfrecord.write_tfrecords(str(tmp_path / ('data-%d.tfrecord' % shard)), records[shard::3])
  pattern = str(tmp_path / 'data-*.tfrecord')
  assert tfdata.get_dataset_metadata(pattern) == ('tfrecord', 3, 1 + 34)
  one_epoch = list(tfdata.parallel_read(pattern, num_epochs=1, seed=0))
  assert sorted(one_epoch) == sorted(records)
  shard_of = {r: i % 3 for i, r in enumerate(records)}
  assert len({shard_of[r] for r in one_epoch[:3]}) == 3                  # one record from every shard in turn
  sequential = list(tfdata.parallel_read(pattern, num_readers=1, num_epochs=1, seed=0))
  assert len({shard_of[r] for r in sequential[:30]}) == 1                # a single reader drains shard after shard
  two_epochs = list(tfdata.parallel_read(pattern, num_epochs=2, seed=1))
  assert len(two_epochs) == 200
  forever = tfdata.parallel_read(pattern)
  assert len([next(forever) for _ in range(350)]) == 350
  feature_spec, label_spec = _pose_env_specs()
  batches = [records[:4], records[4:10]]
  parsed = list(tfdata.serialized_to_parsed(batches, feature_spec, label_spec))
  assert parsed[0][0].action.pose.shape == (4, 2) and parsed[1][1].reward.shape == (6, 1)
  np.testing.assert_array_equal(parsed[1][0].action.pose, GOLDEN['pose'][4:10])


def test_compress_decompress_fns():
  """utils/tfdata.py:546-626: only the tensors with data_format 'jpeg' are touched."""
  spec = utils.TensorSpecStruct(image=TSPEC((32, 48, 3), dtypes.float32, 'image', data_format='jpeg'),
                                depth=TSPEC((32, 48, 1), dtypes.uint8, 'depth', data_format='jpeg'),
                                pose=TSPEC((2,), dtypes.float32, 'pose'))
  rng = np.random.RandomState(0)
  smooth = np.linspace(0, 1, 32 * 48 * 3, dtype=np.float32).reshape(1, 32, 48, 3).repeat(2, 0)
  features = {'image': smooth.copy(), 'depth': (smooth[..., :1] * 255).astype(np.uint8), 'pose': rng.uniform(size=(2, 2))}
  compress = tfdata.create_compress_fn(spec, None, quality=95)
  packed, labels = compress(dict(features))
  assert labels is None and packed['image'].dtype == object and packed['image'][0][:2] == b'\xff\xd8'
  np.testing.assert_array_equal(packed['pose'], features['pose'])
  restored, _ = tfdata.create_decompress_fn(spec, None)(dict(packed))
  assert restored['image'].shape == (2, 32, 48, 3) and restored['image'].dtype == np.float32
  assert restored['depth'].shape == (2, 32, 48, 1) and restored['depth'].dtype == np.uint8
  assert np.abs(restored['image'] - features['image']).max() < 0.05
  assert np.abs(restored['depth'].astype(np.int32) - features['depth'].astype(np.int32)).max() < 10


def test_map_feed_dict_unsafe():
  spec = utils.TensorSpecStruct(a=TSPEC((2,), dtypes.float32, 'a'), b=TSPEC((1,), dtypes.float32, 'b'))
  out = utils.map_feed_dict_unsafe(spec, {'a': np.zeros((3, 2)), 'b': np.zeros((3, 1)), 'extra': np.ones(1)})
  assert list(out) == ['a', 'b']                     # unknown inputs are dropped (with a warning)
  with pytest.raises((KeyError, AttributeError)):      # a missing input fails on lookup, as in the reference
    utils.map_feed_dict_unsafe(spec, {'a': np.zeros((3, 2))})


@pytest.mark.parametrize('batch_size', [1, 2])
def test_varlen_images_feature_spec(tmp_path, batch_size):
  """utils/tfdata_test.py:262-345: a variable number of PNG images per record, padded to the spec with black frames;
  an image of the wrong size is an error."""
  from tensor2robot_b200.utils import image as image_lib
  h, w, padded = 48, 64, 3
  rng = np.random.RandomState(0)
  image_np = rng.uniform(size=(h, w), high=255).astype(np.int32)
  png = image_lib.numpy_to_image_string(image_np, 'png')
  path = str(tmp_path / 'test.tfrecord')
  oracle.write_tfrecords(path, [oracle.make_example({'varlen_images': [png]}),
                                oracle.make_example({'varlen_images': [png, png]})])
  feature_spec = utils.TensorSpecStruct()
  feature_spec.varlen_images = TSPEC(shape=(padded, h, w, 1), dtype=dtypes.uint8, name='varlen_images', data_format='png',
                                     varlen_default_value=0)
  batches = [list(tfdata.parallel_read(path, num_epochs=1, num_readers=1))[:batch_size]]
  (features,) = list(tfdata.serialized_to_parsed(batches, feature_spec, None))
  black = np.zeros((h, w))
  want = np.stack([np.stack([image_np, black, black]), np.stack([image_np, image_np, black])])[:batch_size, ..., None]
  assert features.varlen_images.shape == (batch_size, padded, h, w, 1)
  np.testing.assert_array_equal(features.varlen_images, want)
  # an image whose size differs from the spec
  big = image_lib.numpy_to_image_string(np.ones((2 * h, 2 * w)) * 255, 'png')
  bad_path = str(tmp_path / 'bad.tfrecord')
  oracle.write_tfrecords(bad_path, [oracle.make_example({'varlen_images': [big]}),
                                    oracle.make_example({'varlen_images': [png, big]})])
  bad = [list(tfdata.parallel_read(bad_path, num_epochs=1, num_readers=1))[:batch_size]]
  with pytest.raises(ValueError):
    list(tfdata.serialized_to_parsed(bad, feature_spec, None))


def test_compress_decompress_on_the_fixture():
  """utils/tfdata_test.py:100-141: parse, compress (quality 100), decompress: the frames agree to one decimal."""
  feature_spec = utils.TensorSpecStruct(state=TSPEC((64, 64, 3), dtypes.uint8, 'state/image', data_format='jpeg'),
                                        action=TSPEC((2,), dtypes.bfloat16, 'pose'))
  label_spec = utils.TensorSpecStruct(reward=TSPEC((), dtypes.float32, 'reward'))
  records = list(tfdata.parallel_read(FIXTURE, num_epochs=1))[:5]
  (features, labels), = list(tfdata.serialized_to_parsed([records], feature_spec, label_spec))
  assert features.state.shape == (5, 64, 64, 3)
  original = np.array(features.state)
  flat_f, flat_l = utils.flatten_spec_structure(features), utils.flatten_spec_structure(labels)
  packed, _ = tfdata.create_compress_fn(feature_spec, label_spec, quality=100)(dict(flat_f.items()), dict(flat_l.items()))
  restored, _ = tfdata.create_decompress_fn(feature_spec, label_spec)(packed, dict(flat_l.items()))
  assert restored['state'].shape == (5, 64, 64, 3)
  np.testing.assert_almost_equal(original.astype(np.float32) / 255, restored['state'].astype(np.float32) / 255, decimal=1)


def test_pipelined_input_fn_yields_the_same_batches_in_order(monkeypatch):
  """default_input_fn_tmpl parses up to PARSE_PIPELINE_DEPTH batches concurrently (the reference's num_parallel_calls,
  utils/tfdata.py:629-689); the stream of batches - order, contents, drop_remainder, end of data while parses are still
  in flight (the record mappings must outlive the generator of pointers) - equals the one-at-a-time pipeline."""
  feature_spec, label_spec = _pose_env_specs()

  def run(depth, mode):
    monkeypatch.setattr(tfdata, 'PARSE_PIPELINE_DEPTH', depth)
    out = []
    for features, labels in tfdata.default_input_fn_tmpl(FIXTURE, 16, feature_spec, label_spec, mode=mode, seed=3):
      out.append((features.state.image.copy(), features.action.pose.copy(), labels.reward.copy()))
      if len(out) == 9:                      # TRAIN repeats forever
        break
    return out

  for mode in (tfdata.ModeKeys.EVAL, tfdata.ModeKeys.TRAIN):
    serial, piped = run(1, mode), run(2, mode)
    assert len(serial) == len(piped) == (6 if mode == tfdata.ModeKeys.EVAL else 9)   # 100 records: 6 full batches of 16
    for a, b in zip(serial, piped):
      for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
