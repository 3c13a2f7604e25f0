"""Host-side logic of the training step on CPU: the Keras-2 Nadam schedule, the oracle's Nadam restatement against
torch.optim.NAdam, and the data-parallel gradient exchange under gloo (world_size 2)."""
import os

import numpy as np
import pytest

from dsen2_b200 import train
from oracle import train_oracle as to


def test_nadam_schedule_matches_keras_recurrence():
    opt = train.Nadam()
    assert (opt.lr, opt.beta_1, opt.beta_2, opt.epsilon, opt.schedule_decay) == (1e-4, 0.9, 0.999, 1e-8, 0.004)
    ms = 1.0
    for t in range(1, 50):
        s = train.nadam_schedule(t, ms, opt)
        mu_t = 0.9 * (1.0 - 0.5 * 0.96 ** (t * 0.004))
        mu_n = 0.9 * (1.0 - 0.5 * 0.96 ** ((t + 1) * 0.004))
        assert s['mu_t'] == mu_t and s['mu_next'] == mu_n
        assert np.isclose(s['sched_new'], ms * mu_t) and np.isclose(s['sched_next'], ms * mu_t * mu_n)
        assert np.isclose(s['bias2'], 1.0 - 0.999 ** t)
        ms = s['sched_new']


def test_oracle_nadam_equals_torch_nadam():
    import torch
    rng = np.random.RandomState(0)
    p = rng.randn(500)
    pt = torch.tensor(p.copy(), requires_grad=True)
    opt = torch.optim.NAdam([pt], lr=1e-3, betas=(0.9, 0.999), eps=1e-8, momentum_decay=0.004)
    m = np.zeros_like(p); v = np.zeros_like(p); ms = 1.0
    for t in range(1, 8):
        g = rng.randn(500)
        pt.grad = torch.tensor(g.copy())
        opt.step()
        p, m, v, ms = to.nadam_reference(p, g, m, v, t, ms, lr=1e-3)
        np.testing.assert_allclose(p, pt.detach().numpy(), rtol=0, atol=1e-10)


def test_oracle_training_reduces_the_loss():
    rng = np.random.RandomState(1)
    from oracle import dsen2net_oracle as no
    w = no.he_uniform_weights(10, 6, 1, 8, seed=0)
    xs = [rng.rand(2, 4, 8, 8).astype(np.float32), rng.rand(2, 6, 8, 8).astype(np.float32)]
    y = (xs[1] + 0.1).astype(np.float32)
    losses, _ = to.train_steps([(xs, y)] * 20, w, lr=1e-2)
    assert losses[-1] < 0.5 * losses[0]


def _worker(rank, world, port, tmp):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    flat = torch.arange(1000, dtype=torch.float32) * (rank + 1)
    w = train.allreduce_gradients(flat)
    ok = w == world and torch.equal(flat, torch.arange(1000, dtype=torch.float32) * sum(range(1, world + 1)))
    # averaged gradient = what Trainer.apply_gradients(1/world) hands to the Nadam kernel
    avg = flat / w
    ok = ok and torch.allclose(avg, torch.arange(1000, dtype=torch.float32) * (world + 1) / 2)
    if rank == 0:
        np.save(os.path.join(tmp, 'ok.npy'), np.array([ok]))
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_world2_gradient_allreduce(tmp_path):
    import torch.multiprocessing as mp
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert np.load(str(tmp_path / 'ok.npy'))[0]


def _worker_setup(rank, world, port, tmp):
    """What ``python -m torch.distributed.run -m dsen2_b200.supres_train`` does before training, on the gloo backend:
    process group first, rank 0's weights everywhere, equal-length shards.  The ranks are CPU processes: with CUDA visible,
    dist_setup would select device LOCAL_RANK, which a machine with fewer GPUs than ranks does not have."""
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      CUDA_VISIBLE_DEVICES='')
    import torch.distributed as dist
    from dsen2_b200.DSen2Net import s2model
    assert train.dist_setup('gloo') == (rank, world)
    model = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=100 + rank)   # different draws
    before = model.get_weights()[0].copy()
    train.broadcast_weights(model)
    ref = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=100).get_weights()
    same = all(np.array_equal(a, b) for a, b in zip(model.get_weights(), ref))
    changed = rank == 0 or not np.array_equal(before, model.get_weights()[0])
    xs, y = [np.arange(11 * 2).reshape(11, 2), np.arange(11 * 3).reshape(11, 3)], np.arange(11)
    sx, sy = train.shard_training_set(xs, y, rank, world)
    np.save(os.path.join(tmp, 'r%d.npy' % rank), np.array([same and changed, len(sy), len(sx[0]), int(sy[0]), int(sx[1][0, 0])]))
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_world2_distributed_setup_broadcast_and_equal_shards(tmp_path):
    import torch.multiprocessing as mp
    port = 33500 + (os.getpid() % 2000)
    mp.spawn(_worker_setup, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(str(tmp_path / 'r0.npy')), np.load(str(tmp_path / 'r1.npy'))
    assert r0[0] == 1 and r1[0] == 1                  # both replicas hold rank 0's weights
    assert r0[1] == r1[1] == 5 and r0[2] == r1[2] == 5   # 11 samples over 2 ranks: 5 + 5, the odd one is dropped
    assert (r0[3], r1[3]) == (0, 1) and (r0[4], r1[4]) == (0, 3)


def test_dist_setup_without_a_launcher_is_a_no_op():
    env = {k: os.environ.pop(k) for k in ('RANK', 'WORLD_SIZE') if k in os.environ}
    try:
        assert train.dist_setup() == (0, 1)
    finally:
        os.environ.update(env)


def test_to_yaml_describes_the_network():
    import yaml
    from dsen2_b200.DSen2Net import s2model
    m = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=6, feature_size=128)
    d = yaml.safe_load(m.to_yaml())
    cfg = d['config']
    assert cfg['num_layers'] == 6 and cfg['feature_size'] == 128 and cfg['input_shape'] == [[4, None, None], [6, None, None], [2, None, None]]
    convs = [l for l in cfg['layers'] if l['class_name'] == 'Conv2D']
    assert len(convs) == 14 and convs[0]['filters'] == 128 and convs[-1]['filters'] == 2
    assert sum(l['class_name'] == 'Add' for l in cfg['layers']) == 7


def test_allreduce_is_identity_without_a_process_group():
    import torch
    flat = torch.ones(10)
    assert train.allreduce_gradients(flat) == 1 and torch.equal(flat, torch.ones(10))


# ---- callbacks and data-set loaders (host-side bookkeeping around model.fit, supres_train.py:195-230) ------------
class _FakeOpt:
    lr = 1e-4


class _FakeModel:
    def __init__(self):
        self.optimizer = _FakeOpt()
        self.saved = []

    def save_weights(self, path):
        self.saved.append(path)


def test_reduce_lr_on_plateau_follows_the_keras_state_machine():
    from dsen2_b200.callbacks import ReduceLROnPlateau
    m = _FakeModel()
    cb = ReduceLROnPlateau(monitor='val_loss', factor=0.5, patience=2, epsilon=1e-6, cooldown=2, min_lr=3e-5)
    cb.set_model(m)
    cb.on_train_begin()
    lrs = []
    for ep, v in enumerate([1.0, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9]):
        cb.on_epoch_end(ep, {'val_loss': v})
        lrs.append(m.optimizer.lr)
    # improvement at epochs 0,1; plateau -> wait 1,2 -> reduce after epoch 3; cooldown 2 epochs; then patience again
    assert lrs[:3] == [1e-4, 1e-4, 1e-4] and lrs[3] == 5e-5
    assert lrs[4] == 5e-5 and lrs[5] == 5e-5          # cooling down
    assert lrs[7] == 3e-5                              # second reduction clamps at min_lr
    assert lrs[-1] == 3e-5                             # never below min_lr


def test_model_checkpoint_saves_best_only():
    from dsen2_b200.callbacks import ModelCheckpoint
    m = _FakeModel()
    cb = ModelCheckpoint('w_{epoch:02d}.hdf5', monitor='val_loss', save_best_only=True)
    cb.set_model(m)
    for ep, v in enumerate([1.0, 1.2, 0.8, 0.8, 0.7]):
        cb.on_epoch_end(ep, {'val_loss': v})
    assert m.saved == ['w_01.hdf5', 'w_03.hdf5', 'w_05.hdf5']


def test_training_data_loaders(tmp_path):
    from dsen2_b200 import patches
    rng = np.random.RandomState(0)
    root = str(tmp_path) + '/'
    for i, name in enumerate(['A.SAFE', 'B.SAFE']):
        d = tmp_path / 'train' / name
        d.mkdir(parents=True)
        np.save(d / 'data10.npy', rng.rand(5, 4, 8, 8).astype(np.float32) * 2000)
        np.save(d / 'data20.npy', rng.rand(5, 6, 8, 8).astype(np.float32) * 2000)
        np.save(d / 'data20_gt.npy', rng.rand(5, 6, 8, 8).astype(np.float32) * 2000)
    val = np.zeros(10, bool)
    val[[1, 7]] = True
    np.save(tmp_path / 'train' / 'val_index.npy', val)
    train, label, val_tr, val_lb = patches.OpenDataFiles(root, False, 2000)
    assert [a.shape for a in train] == [(8, 4, 8, 8), (8, 6, 8, 8)] and label.shape == (8, 6, 8, 8)
    assert [a.shape for a in val_tr] == [(2, 4, 8, 8), (2, 6, 8, 8)] and val_lb.shape == (2, 6, 8, 8)
    assert train[0].dtype == np.float32 and 0 <= train[0].min() and train[0].max() <= 1.0
    import json
    t = tmp_path / 'test' / 'C.SAFE'
    t.mkdir(parents=True)
    np.save(t / 'data10.npy', rng.rand(4, 4, 32, 32).astype(np.float32))
    np.save(t / 'data20.npy', rng.rand(4, 6, 32, 32).astype(np.float32))
    json.dump([10, 20, 58, 68], open(t / 'roi.json', 'w'))
    tr, size = patches.OpenDataFilesTest(str(t), False, 2000)
    assert size == [48, 48] and len(tr) == 2 and tr[1].shape == (4, 6, 32, 32)


def test_full_model_file_without_optimizer_state(tmp_path):
    """model.save of an uncompiled model: Keras' full-model layout (/model_weights + model_config); load_weights reads it."""
    import json
    from dsen2_b200.DSen2Net import s2model
    from dsen2_b200.hdf5 import File
    shp = ((4, None, None), (6, None, None))
    m = s2model(shp, num_layers=2, feature_size=128, seed=5)
    p = str(tmp_path / 'full.hdf5')
    m.save(p)
    f = File(p)
    assert list(f.keys()) == ['model_weights']
    cfg = json.loads(bytes(f.attrs['model_config']).decode())['config']
    assert cfg['num_layers'] == 2 and cfg['feature_size'] == 128
    assert [bytes(n).decode() for n in f['model_weights'].attrs['layer_names']] == ['conv2d_%d' % (i + 1) for i in range(6)]
    m2 = s2model(shp, num_layers=2, feature_size=128, seed=6)
    m2.load_weights(p)
    for a, b in zip(m.get_weights(), m2.get_weights()):
        assert np.array_equal(a, b)
    with pytest.raises(RuntimeError):
        m2.load_optimizer_weights(p)                    # not compiled


def test_model_checkpoint_full_model_vs_weights_only():
    from dsen2_b200.callbacks import ModelCheckpoint

    class M(_FakeModel):
        def save(self, path):
            self.saved.append('full:' + path)
    for weights_only, want in ((False, ['full:a.hdf5']), (True, ['a.hdf5'])):
        m = M()
        cb = ModelCheckpoint('a.hdf5', save_weights_only=weights_only)
        cb.set_model(m)
        cb.on_epoch_end(0, {'val_loss': 1.0})
        assert m.saved == want
