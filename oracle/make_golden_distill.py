"""Pins oracle/distill_oracle.py (SURVEY.md section 8 a16-a18) against the UNMODIFIED reference: drives the reference's
own training iteration on the CPU -- SirenMorpher03TrainerArgs / SirenFaceMorpher00TrainerArgs build the computation
protocol, the SumLoss of (time-weighted | masked) L1 terms, the Adam optimizer and SirenMorpherTrainingProtocol03, whose
run_training_iteration (siren_morpher_protocols_03.py:178-214) is called once -- with a stub teacher poser that
returns fixed tensors, and records loss terms, the flat gradient and the parameters after the optimizer step.

Build container only:  python -m oracle.make_golden_distill   ->  tests/golden/distill_lambda00.npz
TEST INFRASTRUCTURE (the GPU box has no /root/reference; the fixture travels instead)."""
import os
import sys

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader, synth  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
BODY_WEIGHTS = (1.0, 0.5, 2.0, 0.25)       # full_blended, full_warped, full_grid_change, full_color_change
LR = 1e-4
GRAD_STRIDE = 37


def distill_inputs():
    """Deterministic inputs shared by the generator and the tests (no teacher network involved: the teacher's role is
    played by fixed smooth tensors, so that the fixture pins the student / loss / optimizer arithmetic alone)."""
    n = 1
    image = synth.synthetic_image(11, n)
    pose = synth.random_poses(n, seed=4)
    smooth = lambda seed, c, amp=1.0: (synth.synthetic_image(seed, n)[:, :c] * amp).contiguous()   # noqa: E731
    body = dict(image=image, pose=pose, t_posed=smooth(12, 4), t_warped=smooth(13, 4), t_grid=smooth(14, 2, 0.05))
    face_posed = smooth(15, 4)[:, :, 100:292, 150:342].contiguous()          # stands for mode_12 output 0: [n,4,192,192]
    g = torch.Generator().manual_seed(5)
    mask = (torch.rand(n, 1, 128, 128, generator=g) > 0.7).float().repeat(1, 4, 1, 1).contiguous()
    face = dict(pose=pose, posed_face=face_posed, mask=mask)
    return body, face


class _StubPoser:
    """Quacks like the teacher inside the protocols: get_posing_outputs(image, pose) -> fixed list, to(device)."""

    def __init__(self, outputs):
        self.outputs = outputs

    def get_posing_outputs(self, image, pose):
        return self.outputs

    def to(self, device):
        return self


def _flat(tensors):
    return torch.cat([t.detach().reshape(-1) for t in tensors])


def reference_body_step(student_sd, inp):
    ref_loader.load()
    from tha4.nn.siren.morpher import siren_morpher_03_trainer as T
    outs = [None] * 33
    outs[0], outs[2], outs[3], outs[5] = inp['t_posed'], inp['t_warped'], inp['t_grid'], inp['image']
    outs[1] = torch.zeros(1, 1, 512, 512)
    weights = {T.LossTerm.full_blended: BODY_WEIGHTS[0], T.LossTerm.full_warped: BODY_WEIGHTS[1],
               T.LossTerm.full_grid_change: BODY_WEIGHTS[2], T.LossTerm.full_color_change: BODY_WEIGHTS[3]}
    args = T.SirenMorpher03TrainerArgs(character_file_name='', pose_dataset_file_name='',
                                       training_phases=T.TrainingPhases([T.TrainingPhase(100_000, LR, T.LossWeights(weights))]),
                                       poser_func=lambda: _StubPoser(outs))
    module = _load_student('body_morpher', student_sd)
    return _run_iteration(args, T.KEY_MODULE, module, [inp['image'], inp['pose'], torch.zeros(1, 4, 512, 512)])


def reference_face_step(student_sd, inp):
    ref_loader.load()
    from tha4.nn.siren.face_morpher import siren_face_morpher_00_trainer as T
    outs = [inp['posed_face']] + [None] * 21
    args = T.SirenFaceMorpher00TrainerArgs(character_file_name='', face_mask_file_name='', pose_dataset_file_name='',
                                           poser_func=lambda: _StubPoser(outs), base_learning_rate=LR)
    module = _load_student('face_morpher', student_sd)
    return _run_iteration(args, T.KEY_MODULE, module, [torch.zeros(1, 4, 512, 512), inp['pose'], inp['mask']])


def _load_student(name, sd):
    import contextlib
    import io
    from tha4.poser.modes import mode_14
    with contextlib.redirect_stdout(io.StringIO()):
        m = mode_14.load_face_morpher(None) if name == 'face_morpher' else mode_14.load_body_morpher(None)
    m.load_state_dict(sd, strict=True)
    return m


def _run_iteration(args, key_module, module, batch):
    protocol = args.get_training_protocol(world_size=1)
    loss = args.get_loss()
    optimizer = args.get_optimizer_factories()[key_module].create(module.parameters())
    lr = protocol.get_learning_rate(0)[key_module]
    for group in optimizer.param_groups:
        group['lr'] = lr
    logged = {}

    def create_log_func(prefix, examples):
        def log(name, value):
            logged[name] = value
        return log

    params = list(module.parameters())
    protocol.run_training_iteration(batch, 0, {key_module: module}, {}, {key_module: optimizer}, {key_module: loss},
                                    create_log_func, torch.device('cpu'))
    return dict(logged=logged, lr=lr, grad=_flat([p.grad for p in params]), params_after=_flat(params))


def main():
    torch.set_num_threads(synth.FIXTURE_THREADS)
    torch.manual_seed(0)
    real = {k: torch.load(os.path.join(GOLDEN, 'data', 'lambda_00_%s.pt' % k), map_location='cpu') for k in ('face_morpher', 'body_morpher')}
    body_in, face_in = distill_inputs()
    out = {}
    for name, res in (('body', reference_body_step(real['body_morpher'], body_in)), ('face', reference_face_step(real['face_morpher'], face_in))):
        print(name, 'reference iteration logged:', {k: round(v, 6) for k, v in res['logged'].items()}, 'lr', res['lr'])
        for k, v in res['logged'].items():
            out['%s_log_%s' % (name, k)] = numpy.float64(v)
        out['%s_lr' % name] = numpy.float64(res['lr'])
        g, p = res['grad'].double(), res['params_after'].double()
        out['%s_grad_sub' % name] = res['grad'][::GRAD_STRIDE].numpy()
        out['%s_grad_stats' % name] = numpy.array([g.norm().item(), g.sum().item(), g.abs().max().item(), float(g.numel())])
        out['%s_params_after_sub' % name] = res['params_after'][::GRAD_STRIDE].numpy()
        out['%s_params_after_stats' % name] = numpy.array([p.norm().item(), p.sum().item()])
    numpy.savez_compressed(os.path.join(GOLDEN, 'distill_lambda00.npz'), **out)
    print('written', os.path.join(GOLDEN, 'distill_lambda00.npz'))


if __name__ == '__main__':
    main()
