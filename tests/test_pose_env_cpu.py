"""CPU-side checks of the pose_env port (BASELINE config C1): model / preprocessor specs as in
research/pose_env/pose_env_models.py, the reference fixture parsed through those specs, and the float64 network
oracle (oracle/vision_layers.py) cross-checked against independent restatements."""
import os

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, 'golden', 'pose_env_test_data.tfrecord')
GOLDEN = np.load(os.path.join(HERE, 'golden', 'pose_env_golden.npz'))


@pytest.fixture(autouse=True)
def _host_image_decoder(monkeypatch):
  """The host decoder (numpy out) on every machine: 'auto' picks the device decoder where a GPU is present, and
  tests/test_jpeg.py checks that one against this one."""
  from tensor2robot_b200.utils import tfdata
  monkeypatch.setattr(tfdata, 'IMAGE_DECODER', 'host')


def test_model_specs():
  from tensor2robot_b200.research.pose_env import pose_env_models as pm
  from tensor2robot_b200.utils import dtypes
  reg = pm.PoseEnvRegressionModel()
  f = reg.get_feature_specification('train')
  assert f.state.shape == (64, 64, 3) and f.state.dtype == dtypes.float32 and f.state.name == 'state/image'
  assert reg.preprocessor.get_in_feature_specification('train').state.dtype == dtypes.uint8
  l = reg.get_label_specification('train')
  assert l.target_pose.shape == (2,) and l.reward.shape == (1,) and reg.action_size == 2
  mc = pm.PoseEnvContinuousMCModel()
  f = mc.get_feature_specification('train')
  assert f.state.image.shape == (64, 64, 3) and f.action.pose.shape == (2,) and f.action.pose.name == 'pose'
  assert mc.get_label_specification('train').reward.shape == ()
  pin = mc.preprocessor.get_in_feature_specification('train')
  assert pin['state/image'].dtype == dtypes.uint8 and pin['state/image'].data_format == 'jpeg'
  packed = mc.pack_features(np.zeros((64, 64, 3), np.uint8), None, 0, np.zeros((5, 2), np.float32))
  assert packed.state.shape == (1, 64, 64, 3) and packed.action.shape == (5, 2)


def test_fixture_parses_through_model_specs():
  from tensor2robot_b200.input_generators import default_input_generator as gens
  from tensor2robot_b200.research.pose_env import pose_env_models as pm
  from tensor2robot_b200.utils import train_eval
  model = pm.PoseEnvContinuousMCModel()
  gen = gens.DefaultRecordInputGenerator(batch_size=4, file_patterns=FIXTURE)
  train_eval.provide_input_generator_with_model_information(gen, model, 'eval')
  features, labels = next(iter(gen.create_dataset_input_fn('eval')()))
  assert features['state/image'].shape == (4, 64, 64, 3) and features['state/image'].dtype == np.uint8
  np.testing.assert_array_equal(features['action/pose'], GOLDEN['pose'][:4])
  np.testing.assert_array_equal(labels['reward'], GOLDEN['reward'][:4, 0])
  np.testing.assert_array_equal(features['state/image'][:, :2, :2], GOLDEN['image_corner'][:4])


def test_network_oracle_building_blocks():
  from oracle import spatial_softmax as ss
  from oracle import vision_layers as o
  rng = np.random.RandomState(0)
  x = rng.standard_normal((3, 9, 7, 5))
  np.testing.assert_allclose(o.layer_norm(torch.from_numpy(x), torch.ones(5, dtype=torch.float64), torch.zeros(5, dtype=torch.float64)).numpy(),
                             torch.nn.functional.layer_norm(torch.from_numpy(x), (9, 7, 5), eps=1e-12).numpy(), atol=1e-12)
  points, _ = ss.build_spatial_softmax(x)                      # float32 positions / outputs like the reference
  np.testing.assert_allclose(o.spatial_softmax(torch.from_numpy(x)).numpy(), points, atol=1e-6)
  # the action merge tiles the whole image batch (tf.tile), it does not repeat each image
  w = {'q_func/q_features/fully_connected/weights': torch.zeros(2, 32, dtype=torch.float64),
       'q_func/q_features/fully_connected/biases': torch.zeros(32, dtype=torch.float64)}
  for i, s in enumerate(('Conv', 'Conv_1', 'Conv_2')):
    w['q_func/q_features/%s/weights' % s] = torch.from_numpy(rng.standard_normal((3, 3, 3 if i == 0 else 32, 32)))
    w['q_func/q_features/%s/LayerNorm/gamma' % s] = torch.ones(32, dtype=torch.float64)
    w['q_func/q_features/%s/LayerNorm/beta' % s] = torch.zeros(32, dtype=torch.float64)
  k = 7 * 7 * 32
  for i in (1, 2):
    w['q_func/Stack/fully_connected_%d/weights' % i] = torch.from_numpy(rng.standard_normal((k, 100)) * 0.05)
    w['q_func/Stack/fully_connected_%d/biases' % i] = torch.zeros(100, dtype=torch.float64)
    k = 100
  w['q_func/fully_connected/weights'] = torch.from_numpy(rng.standard_normal((100, 1)))
  w['q_func/fully_connected/biases'] = torch.zeros(1, dtype=torch.float64)
  img = torch.from_numpy(rng.uniform(size=(2, 64, 64, 3)))
  q = o.mc_critic_q(img, torch.zeros(4, 2, dtype=torch.float64), w)
  assert q.shape == (4,)
  np.testing.assert_allclose(q[:2].numpy(), q[2:].numpy(), rtol=1e-12)      # rows 2, 3 are images 0, 1 again
  assert abs(float(q[0] - q[1])) > 0
