"""Replay-writing side (SURVEY 8 F-1): the Example encoder + TFRecordReplayWriter reproduce the reference's own fixture
byte for byte from its parsed contents (features re-inserted in each record's wire order: the python protobuf runtime
that wrote the fixture emits map entries in no canonical order), and episode_to_transitions output parses back through
the model specs."""
import os

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import tfrecord

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, 'golden', 'pose_env_test_data.tfrecord')


@pytest.fixture(autouse=True)
def _host_image_decoder(monkeypatch):
  """The host decoder (numpy out) on every machine: 'auto' picks the device decoder where a GPU is present, and
  tests/test_jpeg.py checks that one against this one."""
  from tensor2robot_b200.utils import tfdata
  monkeypatch.setattr(tfdata, 'IMAGE_DECODER', 'host')


def _rebuild(parsed):
  from tensor2robot_b200.utils import example_proto as ep
  features = {}
  for key, (kind, values) in parsed.items():      # wire order of this record (protobuf map order is not canonical)
    features[key] = {'bytes': ep.bytes_feature, 'float': ep.float_feature, 'int64': ep.int64_feature}[kind](values)
  return ep.Example(features=features)


def test_fixture_reproduced_byte_for_byte(tmp_path):
  from tensor2robot_b200.utils import writer
  records = tfrecord.read_tfrecords(FIXTURE)
  examples = [_rebuild(tfrecord.parse_example(r)) for r in records]
  for rec, ex in zip(records, examples):
    assert ex.SerializeToString() == rec
  w = writer.TFRecordReplayWriter()
  with pytest.raises(ValueError):
    w.write(examples)
  w.open(str(tmp_path / 'sub' / 'replay'))
  with pytest.raises(ValueError):
    w.open(str(tmp_path / 'other'))
  w.write(examples[:40])
  w.write(examples[40:])
  w.close()
  with pytest.raises(ValueError):
    w.close()
  with open(FIXTURE, 'rb') as f, open(str(tmp_path / 'sub' / 'replay.tfrecord'), 'rb') as g:
    assert f.read() == g.read()


@settings(max_examples=60, deadline=None)
@given(st.lists(st.integers(min_value=-2**63, max_value=2**63 - 1), max_size=6),
       st.lists(st.floats(width=32, allow_nan=False), max_size=6), st.lists(st.binary(max_size=40), max_size=3))
def test_encoder_round_trips_through_the_oracle_parser(ints, floats, blobs):
  from tensor2robot_b200.utils import example_proto as ep
  ex = ep.Example({'i': ep.int64_feature(ints), 'f': ep.float_feature(floats), 'b': ep.bytes_feature(blobs)})
  parsed = tfrecord.parse_example(ex.SerializeToString())
  assert [int(v) for v in parsed['i'][1]] == ints if ints else len(parsed.get('i', (None, []))[1]) == 0
  got_f = parsed.get('f', (None, []))[1]
  assert np.array_equal(np.asarray(got_f, np.float32), np.asarray(floats, np.float32))
  assert list(parsed.get('b', (None, []))[1]) == blobs
  # the oracle's own encoder agrees on the bytes (same insertion order)
  if ints and floats and blobs:
    assert ex.SerializeToString() == tfrecord.make_example({'i': ints, 'f': floats, 'b': blobs})


def test_episode_to_transitions_feeds_the_models(tmp_path):
  from tensor2robot_b200.input_generators import default_input_generator as gens
  from tensor2robot_b200.research.pose_env import episode_to_transitions as e2t
  from tensor2robot_b200.research.pose_env import pose_env_models as pm
  from tensor2robot_b200.utils import train_eval
  from tensor2robot_b200.utils import writer
  rng = np.random.RandomState(0)
  episodes = []
  for _ in range(3):
    obs = np.kron(rng.randint(0, 256, (8, 8, 3)), np.ones((8, 8, 1))).astype(np.uint8)     # blocky 64x64 frame
    episodes.append([(obs, rng.uniform(-1, 1, (1, 2)).astype(np.float32), float(-rng.uniform()), obs, True,
                      {'target_pose': rng.uniform(-1, 1, 2).astype(np.float32)})])
  w = writer.TFRecordReplayWriter()
  w.open(str(tmp_path / 'replay'))
  for episode in episodes:
    w.write(e2t.episode_to_transitions_pose_toy(episode))
  w.close()
  model = pm.PoseEnvRegressionModel()
  gen = gens.DefaultRecordInputGenerator(batch_size=3, file_patterns=str(tmp_path / 'replay.tfrecord'))
  train_eval.provide_input_generator_with_model_information(gen, model, 'eval')
  features, labels = next(iter(gen.create_dataset_input_fn('eval')()))
  assert features['state'].shape == (3, 64, 64, 3)
  want = np.stack([e[0][5]['target_pose'] for e in episodes])
  np.testing.assert_array_equal(labels['target_pose'], want)
  np.testing.assert_allclose(labels['reward'][:, 0], [e[0][2] for e in episodes], rtol=1e-7)
  assert np.abs(features['state'].astype(np.int32) - np.stack([e[0][0] for e in episodes]).astype(np.int32)).mean() < 16   # JPEG q90 with 4:2:0 chroma on saturated blocks
