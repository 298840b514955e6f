"""Record, from the UNMODIFIED reference, what the reference-pinned tests compare against, so that they run from the
repository alone:

  tests/golden/reference_posers.npz      mode_07 / mode_12 / mode_14 outputs (synthetic image 3, pose seed 77) and
                                         the state_dict layout of every network
  tests/golden/reference_distill.npz     gradient and post-Adam parameters of the reference training iteration
  tests/golden/reference_image_io.npz    the reference's PNG loader and its output / display conversions
  tests/golden/reference_pins.json       pose schema, poser getters, training schedules and the files the
                                         reference's training-state loader requires

Tensors are stored as a fixed spread-out sample of their elements (spread()) together with mean / mean|x| / max|x|
over the full tensor, so that the fixtures stay small; poser outputs also keep the mean of every 32x32 tile
(tile_means()), so that an error confined to a small patch still shows.

Needs the reference checkout:  THA4_REFERENCE_ROOT=<checkout> python -m oracle.make_golden_pins
"""
import contextlib
import io
import json
import os
import sys
import tempfile

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader, synth  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
SPREAD_STEP = 104729                  # a prime: coprime with every tensor size here, so the sample has no repeats
PROBE_EXAMPLES = [0, 199_999, 200_000, 200_001, 1_299_999, 1_300_000, 1_499_992, 2_000_000] + list(range(0, 1_600_000, 50_000))
FACE_PROBE_EXAMPLES = [0, 199_999, 200_000, 499_999, 500_000, 799_999, 800_000, 999_999, 5_000_000]


def poser_inputs():
    return synth.synthetic_image(3, 1)[0], synth.random_poses(1, seed=77)[0]


def display_input():
    return synth.synthetic_image(3, 1)[0] * 1.05


def spread(t, n):
    """n elements of t (all of them if it has fewer): flat indices (k * SPREAD_STEP + 7) mod numel, k = 0 .. n - 1."""
    flat = torch.as_tensor(t).reshape(-1)
    if flat.numel() <= n:
        return flat
    return flat[(torch.arange(n, dtype=torch.int64) * SPREAD_STEP + 7) % flat.numel()]


def tile_means(t, tile=32):
    """Mean of every tile x tile block of each [H, W] plane of an [N, C, H, W] tensor (float64 sums, stored float32)."""
    n, c, h, w = t.shape
    return t.double().reshape(n, c, h // tile, tile, w // tile, tile).mean(dim=(3, 5)).float().numpy()


def stats(t):
    t = t.double()
    return numpy.array([t.mean().item(), t.abs().mean().item(), t.abs().max().item()])


def poser_outputs(mods):
    img, pose = poser_inputs()
    out = {}
    for mode, grp in (('mode_07', 'teacher'), ('mode_12', 'teacher'), ('mode_14', 'student')):
        outs = ref_loader.reference_poser(mode, mods[grp]).get_posing_outputs(img, pose)
        out['%s_count' % mode] = numpy.int64(len(outs))
        for i, t in enumerate(outs):
            out['%s_o%02d' % (mode, i)] = spread(t, 256).numpy()
            out['%s_o%02d_shape' % (mode, i)] = numpy.array(t.shape)
            out['%s_o%02d_stats' % (mode, i)] = stats(t)
            out['%s_o%02d_tiles' % (mode, i)] = tile_means(t)
    return out


def layouts(mods):
    """One 'key shape' line per state_dict entry, in order, for every network."""
    return {'layout_%s_%s' % (grp, name): numpy.array('\n'.join('%s %s' % (k, list(v.shape)) for k, v in m.state_dict().items()))
            for grp in ('teacher', 'student') for name, m in mods[grp].items()}


def distill_pins():
    from oracle import make_golden_distill as M
    real = {k: torch.load(os.path.join(GOLDEN, 'data', 'lambda_00_%s.pt' % k), map_location='cpu') for k in ('face_morpher', 'body_morpher')}
    body_in, face_in = M.distill_inputs()
    out = {}
    for net, res in (('body', M.reference_body_step(real['body_morpher'], body_in)), ('face', M.reference_face_step(real['face_morpher'], face_in))):
        out['%s_logged_loss' % net] = numpy.float64(res['logged']['loss'])
        out['%s_grad_sub' % net] = spread(res['grad'], 4096).numpy()
        out['%s_grad_absmax' % net] = numpy.float64(res['grad'].abs().max().item())
        out['%s_params_after_sub' % net] = spread(res['params_after'], 4096).numpy()
        out['%s_numel' % net] = numpy.int64(res['grad'].numel())
    return out


def image_io_pins():
    from tha4.shion.base.image_util import extract_pytorch_image_from_filelike
    from tha4.image_util import convert_linear_to_srgb, convert_output_image_from_torch_to_numpy
    png = os.path.join(GOLDEN, 'data', 'lambda_00.png')
    loaded = extract_pytorch_image_from_filelike(png, scale=2.0, offset=-1.0, premultiply_alpha=True, perform_srgb_to_linear=True)
    out = synth.synthetic_image(3, 1)[0]
    x = display_input()
    o = torch.clip((x + 1.0) / 2.0, 0.0, 1.0)
    srgb = convert_linear_to_srgb(o)
    rgba8 = torch.from_numpy(convert_output_image_from_torch_to_numpy(out))
    return {'loaded_shape': numpy.array(loaded.shape), 'loaded_sub': spread(loaded, 8192).numpy(), 'loaded_stats': stats(loaded),
            'output_rgba8_shape': numpy.array(rgba8.shape), 'output_rgba8_sub': spread(rgba8, 8192).numpy(),
            'display_srgb_sub': spread(srgb, 8192).numpy(), 'display_srgb_stats': stats(srgb),
            'display_srgb8_sub': spread((255.0 * srgb).permute(1, 2, 0).byte(), 8192).numpy()}


def pose_and_poser_pins(student_mods):
    from tha4.poser.modes.pose_parameters import get_pose_parameters
    params = get_pose_parameters()
    groups = [dict(group_name=g.get_group_name(), arity=g.get_arity(), parameter_index=g.get_parameter_index(),
                   parameter_names=g.get_parameter_names(), category=[g.get_category().name, g.get_category().value],
                   default_value=g.get_default_value(), range=list(g.get_range()), discrete=g.is_discrete())
              for g in params.get_pose_parameter_groups()]
    poser = ref_loader.reference_poser('mode_14', student_mods)
    surface = dict(image_size=poser.get_image_size(), output_length=poser.get_output_length(),
                   num_parameters=poser.get_num_parameters(), dtype=str(poser.get_dtype()))
    return dict(parameter_count=params.get_parameter_count(), groups=groups,
                parameter_names=[params.get_parameter_name(i) for i in range(params.get_parameter_count())], mode_14_poser=surface)


def schedule_pins():
    from tha4.nn.siren.morpher.siren_morpher_03_trainer import LossTerm, LossWeights, TrainingPhase, TrainingPhases
    from tha4.nn.siren.face_morpher.siren_face_morpher_00_trainer import SirenFaceMorpher00TrainerArgs, KEY_MODULE
    from tha4_b200 import training
    # the body table of the distiller config, evaluated by the reference's own lookup classes
    ours = training.body_morpher_training_phases()
    ref = TrainingPhases([TrainingPhase(p.num_examples_upper_bound, p.learning_rate,
                                        LossWeights({t: p.loss_weights[t.name] for t in LossTerm})) for p in ours.phases])
    lr_func = ref.get_learning_rate_func([KEY_MODULE])
    w_funcs = [ref.get_loss_weight_func(t) for t in LossTerm]
    face = SirenFaceMorpher00TrainerArgs('character.png', 'mask.png', 'poses.pt')
    return dict(loss_terms=[t.name for t in LossTerm],
                body=[[n, lr_func(n)[KEY_MODULE], [f(n) for f in w_funcs]] for n in PROBE_EXAMPLES],
                face=[[n, face.get_learning_rate(n)[KEY_MODULE]] for n in FACE_PROBE_EXAMPLES],
                face_total_examples=face.num_training_total_examples)


def training_state_pins():
    """The files DistributedTrainingState.can_load requires of a one-module, one-optimiser, one-rank state: each one
    is checked to be necessary and the set to be sufficient."""
    from tha4.shion.core.training.distrib.distributed_training_states import DistributedTrainingState as S
    names = [os.path.basename(f('')) for f in (S.get_examples_seen_so_far_file_name, lambda p: S.get_module_file_name(p, 'module'),
                                               lambda p: S.get_optimizer_file_name(p, 'module'), lambda p: S.get_rng_state_file_name(p, 0))]
    check = lambda d: S.can_load(d, {'module': None}, {}, {'module': None}, 1)      # noqa: E731
    with tempfile.TemporaryDirectory() as d:
        for n in names:
            open(os.path.join(d, n), 'w').write('24\n')
        assert check(d) and S.get_examples_seen_so_far(d) == 24
        for n in names:
            os.rename(os.path.join(d, n), os.path.join(d, n + '.off'))
            assert not check(d), n
            os.rename(os.path.join(d, n + '.off'), os.path.join(d, n))
    return dict(required_files=sorted(names))


def main():
    torch.set_num_threads(synth.FIXTURE_THREADS)
    torch.set_grad_enabled(False)
    ref_loader.load()
    tsd, ssd = synth.teacher_state_dicts(0), synth.student_state_dicts(0)
    mods = ref_loader.build_reference_modules(tsd, ssd)
    numpy.savez_compressed(os.path.join(GOLDEN, 'reference_posers.npz'), **poser_outputs(mods), **layouts(mods))
    numpy.savez_compressed(os.path.join(GOLDEN, 'reference_image_io.npz'), **image_io_pins())
    pins = dict(pose=pose_and_poser_pins(mods['student']), schedules=schedule_pins(),
                training_state=training_state_pins())
    with open(os.path.join(GOLDEN, 'reference_pins.json'), 'w') as f:
        json.dump(pins, f, indent=1)
        f.write('\n')
    torch.set_grad_enabled(True)
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        distill = distill_pins()
    numpy.savez_compressed(os.path.join(GOLDEN, 'reference_distill.npz'), **distill)
    print('golden fixtures written to', GOLDEN)


if __name__ == '__main__':
    main()
