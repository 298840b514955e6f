"""Generate tests/golden/ fixtures by running the UNMODIFIED reference (imported from /root/reference) on the CPU.

Run in the build container only:  python -m oracle.make_golden
Writes
  tests/golden/data/              lambda_00 character image + shipped student checkpoints (reference data files,
                                  CC-BY-NC image licence copied alongside) -- the GPU box has no /root/reference
  tests/golden/teacher_seed0.npz  mode_07 (33 outputs) on synthetic weights (oracle/synth.py seed 0), 2 poses
  tests/golden/student_lambda00.npz   mode_14 (6 outputs) with the shipped lambda_00 weights + image, 2 poses
  tests/golden/student_seed0.npz  mode_14 on synthetic student weights
Outputs are stored sub-sampled (every 8th pixel from offset 3, all channels) plus per-tensor mean / mean|x| over the
full tensor, so the fixtures stay < 3 MB while still pinning every output tensor.
"""
import os
import shutil
import sys

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader, synth, image_io  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
STRIDE, OFFSET = 8, 3


def subsample(t: torch.Tensor) -> numpy.ndarray:
    return t[:, :, OFFSET::STRIDE, OFFSET::STRIDE].contiguous().numpy()


def pack(outputs_per_pose):
    d = {}
    for p, outs in enumerate(outputs_per_pose):
        for i, t in enumerate(outs):
            d['p%d_o%02d' % (p, i)] = subsample(t)
            d['p%d_o%02d_stats' % (p, i)] = numpy.array([t.double().mean().item(), t.double().abs().mean().item()])
    return d


def main():
    torch.set_num_threads(synth.FIXTURE_THREADS)
    os.makedirs(os.path.join(GOLDEN, 'data'), exist_ok=True)
    ref = ref_loader.REFERENCE_ROOT
    for src, dst in (('data/images/lambda_00.png', 'lambda_00.png'),
                     ('data/images/README.md', 'IMAGE_LICENSE_README.md'),
                     ('data/character_models/lambda_00/face_morpher.pt', 'lambda_00_face_morpher.pt'),
                     ('data/character_models/lambda_00/body_morpher.pt', 'lambda_00_body_morpher.pt')):
        shutil.copyfile(os.path.join(ref, src), os.path.join(GOLDEN, 'data', dst))
    torch.set_grad_enabled(False)
    poses = synth.random_poses(2, seed=1234)

    tsd = synth.teacher_state_dicts(0)
    ssd = synth.student_state_dicts(0)
    mods = ref_loader.build_reference_modules(tsd, ssd)
    img = synth.synthetic_image(0, 1)[0]
    poser = ref_loader.reference_poser('mode_07', mods['teacher'])
    outs = [poser.get_posing_outputs(img, poses[p]) for p in range(2)]
    numpy.savez_compressed(os.path.join(GOLDEN, 'teacher_seed0.npz'), poses=poses.numpy(), **pack(outs))
    poser = ref_loader.reference_poser('mode_14', mods['student'])
    outs = [poser.get_posing_outputs(img, poses[p]) for p in range(2)]
    numpy.savez_compressed(os.path.join(GOLDEN, 'student_seed0.npz'), poses=poses.numpy(), **pack(outs))

    real = {k: torch.load(os.path.join(GOLDEN, 'data', 'lambda_00_%s.pt' % k), map_location='cpu')
            for k in ('face_morpher', 'body_morpher')}
    mods = ref_loader.build_reference_modules(None, real)
    img = image_io.load_rgba_png(os.path.join(GOLDEN, 'data', 'lambda_00.png'))
    # the reference's own loader must agree with the restated one
    ref_loader.load()
    poser = ref_loader.reference_poser('mode_14', mods['student'])
    outs = [poser.get_posing_outputs(img, poses[p]) for p in range(2)]
    numpy.savez_compressed(os.path.join(GOLDEN, 'student_lambda00.npz'), poses=poses.numpy(), **pack(outs))
    print('golden fixtures written to', GOLDEN)


if __name__ == '__main__':
    main()
