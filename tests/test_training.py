"""Checkpoint / resume format, phase schedules and loop gates of tha4_b200/training.py on the CPU (the CUDA context is a
stub: this tests the host logic around the inner loop, exactly like tests/test_distill_gloo.py).

  * schedules pinned against what the reference's own lookup classes returned (tests/golden/reference_pins.json);
  * a saved state has the reference's file names and an optimiser file a real torch.optim.Adam loads;
  * stop + resume reproduces the uninterrupted run BIT FOR BIT on the flat weight / moment buffers."""
import json
import os

import torch

from tha4_b200 import distill, training
from tha4_b200.poser.modes import mode_14


class _StubCtx:
    device = torch.device('cpu')

    def siren_morpher_train_step(self, image, pose, t0, t2, t3, weights, params, grads, want_losses=True):
        w = torch.tensor(list(weights), dtype=torch.float32)
        grads.copy_(torch.sin(params * 3.0 + pose.sum()) * (0.5 + w.sum()))      # depends on weights, pose and parameters
        return [float(pose.sum()), 0.0, 0.0, 0.0]

    def adam_step(self, params, grads, m, v, lr, step, betas=(0.9, 0.999), eps=1e-8, grad_scale=1.0):
        g = grads * grad_scale
        m.mul_(betas[0]).add_(g, alpha=1 - betas[0])
        v.mul_(betas[1]).addcmul_(g, g, value=1 - betas[1])
        denom = v.sqrt() / (1 - betas[1] ** step) ** 0.5 + eps
        params.addcdiv_(m, denom, value=-lr / (1 - betas[0] ** step))


class _StubTeacher:
    def __init__(self): self.ctx = _StubCtx()
    def get_context(self): return self.ctx
    def get_modules(self): return {}
    def get_posing_outputs(self, image, pose): return [image] * 33


def _make_distiller(seed=0):
    student = mode_14.load_body_morpher(None)
    g = torch.Generator().manual_seed(seed)
    for p in student.parameters():
        p.data.copy_(torch.randn(p.shape, generator=g) * 0.1)
    d = distill.BodyMorpherDistiller.__new__(distill.BodyMorpherDistiller)
    d.teacher, d.student, d.ctx = _StubTeacher(), student, _StubCtx()
    d.flat = distill.flatten_parameters(student)
    d.grad, d.exp_avg, d.exp_avg_sq = (torch.zeros_like(d.flat) for _ in range(3))
    d.betas, d.eps, d.step_count, d.group, d.world = (0.9, 0.999), 1e-8, 0, None, 1
    return d


def _make_trainer(prefix, d, per_snapshot=2):
    phases = training.TrainingPhases([
        training.TrainingPhase(8, 1e-3, {'full_warped': 1.0, 'full_grid_change': 1.0}),
        training.TrainingPhase(16, 3e-4, {'full_blended': 2.0, 'full_color_change': 0.5}),
    ])
    poses = torch.rand(10, 45, generator=torch.Generator().manual_seed(3))
    batches = training.PoseBatches(poses, batch_size=1, rank=0, world=1, seed=11)
    image = torch.zeros(1, 4, 8, 8)
    return training.DistillTrainer(prefix, d, phases, batches,
                                   lambda pose, w, lr: d.train_step(image, pose, w, lr, want_losses=False),
                                   per_checkpoint=8, per_snapshot=per_snapshot)


# ------------------------------------------------------------------------------------------------ schedules
def test_body_phase_table_matches_distiller_config():
    ph = training.body_morpher_training_phases()
    assert [p.num_examples_upper_bound for p in ph.phases] == [200_000, 400_000, 600_000, 800_000, 1_300_000, 1_500_000]
    assert [p.learning_rate for p in ph.phases] == [1e-4, 3e-5, 3e-5, 1e-5, 1e-5, 3e-6]
    assert ph.loss_weights(0) == [0.25, 0.25, 0.5, 2.0] and ph.loss_weights(599_999) == [1.0, 2.5, 5.0, 1.0]
    assert ph.loss_weights(800_000) == [10.0, 1.0, 1.0, 1.0] and ph.loss_weights(10 ** 9) == [10.0, 1.0, 1.0, 1.0]
    assert ph.learning_rate(199_999) == 1e-4 and ph.learning_rate(200_000) == 3e-5 and ph.learning_rate(1_499_999) == 3e-6
    assert ph.total_examples() == 1_500_000


def _reference_pins():
    return json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_pins.json')))


def test_schedules_pinned_to_reference_lookup_rules():
    """The body phase table evaluated by the reference's TrainingPhases lookup, and the reference face trainer's own
    learning-rate schedule, at the example counts around every phase boundary (oracle/make_golden_pins.py)."""
    ref = _reference_pins()['schedules']
    ours = training.body_morpher_training_phases()
    assert ref['loss_terms'] == list(distill.LOSS_TERMS)
    for n, lr, weights in ref['body']:
        assert lr == ours.learning_rate(n), n
        assert weights == ours.loss_weights(n), n
    face = training.FaceMorpherSchedule()
    for n, lr in ref['face']:
        assert lr == face.learning_rate(n), n
    assert face.total_examples() == ref['face_total_examples'] and face.loss_weights(0) == [1.0, 20.0]


# ------------------------------------------------------------------------------------------------ files
def test_state_files_have_reference_layout_and_round_trip(tmp_path):
    d = _make_distiller(1)
    image, pose = torch.zeros(1, 4, 8, 8), torch.rand(1, 45)
    for _ in range(3):
        d.train_step(image, pose, [1.0, 1.0, 0.0, 0.0], 1e-3, want_losses=False)
    st = training.DistillTrainingState(d, examples_seen_so_far=24)
    prefix = str(tmp_path / 'snapshot')
    st.save(prefix, 0, lambda: None, lr=1e-3)
    assert sorted(os.listdir(prefix)) == ['examples_seen_so_far.txt', 'module_module.pt', 'optimizer_module.pt', 'rng_state_00000000.pt']
    assert open(prefix + '/examples_seen_so_far.txt').read() == '24\n'
    assert training.can_load(prefix, 1) and not training.can_load(prefix, 2)         # rank 1's RNG file is missing
    # the module file is a plain reference-format state_dict ...
    sd = torch.load(prefix + '/module_module.pt')
    assert list(sd.keys()) == list(d.student.state_dict().keys())
    fresh = mode_14.load_body_morpher(None, sd)
    # ... and the optimiser file loads into a real torch.optim.Adam over that module's parameters
    opt = torch.optim.Adam(fresh.parameters(), lr=1.0)
    opt.load_state_dict(torch.load(prefix + '/optimizer_module.pt'))
    assert opt.param_groups[0]['lr'] == 1e-3 and opt.param_groups[0]['betas'] == (0.9, 0.999)
    off = 0
    for p in fresh.parameters():
        s = opt.state[p]
        assert float(s['step']) == 3.0
        assert torch.equal(s['exp_avg'].reshape(-1), d.exp_avg[off:off + p.numel()])
        assert torch.equal(s['exp_avg_sq'].reshape(-1), d.exp_avg_sq[off:off + p.numel()])
        off += p.numel()
    # round trip into a different distiller
    d2 = _make_distiller(2)
    st2 = training.DistillTrainingState(d2)
    st2.load(prefix, 0)
    assert st2.examples_seen_so_far == 24 and d2.step_count == 3
    assert torch.equal(d2.flat, d.flat) and torch.equal(d2.exp_avg, d.exp_avg) and torch.equal(d2.exp_avg_sq, d.exp_avg_sq)
    # the reference's own check accepts the directory: every file its can_load requires is there, and its reader
    # (int of the first line) gets the count back
    for name in _reference_pins()['training_state']['required_files']:
        assert os.path.isfile(os.path.join(prefix, name)), name
    assert int(open(prefix + '/examples_seen_so_far.txt').readlines()[0]) == 24


def test_pose_batches_follow_distributed_sampler_and_examples_seen():
    poses = torch.arange(11 * 45, dtype=torch.float32).reshape(11, 45)
    world, batch = 2, 2
    streams = [training.PoseBatches(poses, batch, r, world, seed=5) for r in range(world)]
    assert streams[0].epoch_size == 8                      # 11 -> 10 (world) -> 8 (global batch 4)
    from torch.utils.data import DistributedSampler
    for epoch in range(2):
        for r in range(world):
            sampler = DistributedSampler(list(range(11)), num_replicas=world, rank=r, shuffle=True, seed=5, drop_last=True)
            sampler.set_epoch(epoch)
            idx = list(iter(sampler))
            for it in range(2):
                got = streams[r].get(epoch * 8 + it * batch * world)
                assert torch.equal(got, poses[idx[it * batch:(it + 1) * batch]]), (epoch, r, it)


# ------------------------------------------------------------------------------------------------ loop gates
def test_trainer_gates_and_resume_equals_uninterrupted_run(tmp_path):
    # uninterrupted: 16 examples, checkpoints at 8 and 16, snapshots every 2
    d_full = _make_distiller(0)
    t_full = _make_trainer(str(tmp_path / 'full'), d_full)
    assert t_full.train() == 16
    assert sorted(os.listdir(str(tmp_path / 'full' / 'checkpoint'))) == ['0000', '0001', '0002']
    assert training.read_examples_seen_so_far(t_full.checkpoint_prefix(1)) == 8
    assert training.read_examples_seen_so_far(t_full.checkpoint_prefix(2)) == 16
    assert training.read_examples_seen_so_far(t_full.snapshot_prefix()) == 16
    assert d_full.step_count == 16

    # stopped after 5 iterations (last snapshot at 4 examples), then resumed by a NEW process' worth of objects
    d_a = _make_distiller(0)
    t_a = _make_trainer(str(tmp_path / 'resumed'), d_a)
    assert t_a.train(max_iterations=5) == 5
    assert training.read_examples_seen_so_far(t_a.snapshot_prefix()) == 4
    d_b = _make_distiller(99)                                  # different initial weights: everything must come from the files
    t_b = _make_trainer(str(tmp_path / 'resumed'), d_b)
    assert t_b.train() == 16
    assert d_b.step_count == 16
    assert torch.equal(d_b.flat, d_full.flat), 'resumed weights differ from the uninterrupted run'
    assert torch.equal(d_b.exp_avg, d_full.exp_avg) and torch.equal(d_b.exp_avg_sq, d_full.exp_avg_sq)
    # the phase switch at 8 examples happened in both (different lr and loss weights feed the stub gradient)
    d_c = _make_distiller(0)
    t_c = _make_trainer(str(tmp_path / 'target8'), d_c)
    assert t_c.train(target_checkpoint_examples=8) == 8
    sd8 = torch.load(t_full.checkpoint_prefix(1) + '/module_module.pt')
    assert torch.equal(torch.cat([v.reshape(-1) for v in sd8.values()]), d_c.flat)
    # a finished run is not re-run: the newest state already satisfies the target
    before = d_b.flat.clone()
    assert _make_trainer(str(tmp_path / 'resumed'), d_b).train() == 16 and torch.equal(d_b.flat, before)
