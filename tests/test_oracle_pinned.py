"""Pins the CPU oracle (oracle/tha4_oracle.py, oracle/gridsample_ref.c) to the reference, through the committed golden
fixtures that oracle/make_golden.py, oracle/make_golden_distill.py and oracle/make_golden_pins.py recorded by running the
unmodified reference on seeded weights / the shipped lambda_00 student: sampled output tensors with full-tensor
statistics, the state_dict key/shape layout of every network, the pose schema, the image conversions and the
training schedules.
"""
import ctypes
import json
import os

import numpy
import pytest
import torch
import torch.nn.functional as F

from oracle import image_io, synth, tha4_oracle as O
from oracle.make_golden_pins import display_input, poser_inputs, spread, stats, tile_means

STRIDE, OFFSET = 8, 3


@pytest.fixture(autouse=True, scope='module')
def _fixture_thread_count():
    """The fixtures were recorded with synth.FIXTURE_THREADS CPU threads; the oracle runs with the same count on every
    host, because the thread count moves its outputs by ~1e-5."""
    before = torch.get_num_threads()
    torch.set_num_threads(synth.FIXTURE_THREADS)
    yield
    torch.set_num_threads(before)


def _check_against_golden(npz, outputs_per_pose, tol):
    for p, outs in enumerate(outputs_per_pose):
        for i, t in enumerate(outs):
            g = npz['p%d_o%02d' % (p, i)]
            got = t[:, :, OFFSET::STRIDE, OFFSET::STRIDE].numpy()
            assert got.shape == g.shape
            assert numpy.abs(got - g).max() <= tol, (p, i)
            stats = npz['p%d_o%02d_stats' % (p, i)]
            assert abs(t.double().mean().item() - stats[0]) <= tol
            assert abs(t.double().abs().mean().item() - stats[1]) <= tol


def test_teacher_oracle_matches_golden(golden_dir, teacher_sds):
    npz = numpy.load(os.path.join(golden_dir, 'teacher_seed0.npz'))
    poses = torch.from_numpy(npz['poses'])
    assert torch.equal(poses, synth.random_poses(2, 1234))
    img = synth.synthetic_image(0, 1)[0]
    with torch.no_grad():
        outs = [O.mode_07_outputs(teacher_sds, img, poses[p]) for p in range(2)]
    assert len(outs[0]) == 33
    # same torch build => bit-identical; 1e-5 leaves room for a different CPU vector ISA on another host
    _check_against_golden(npz, outs, 1e-5)


def test_student_oracle_matches_golden(golden_dir, student_sds, lambda00_sds):
    with torch.no_grad():
        npz = numpy.load(os.path.join(golden_dir, 'student_seed0.npz'))
        poses = torch.from_numpy(npz['poses'])
        img = synth.synthetic_image(0, 1)[0]
        _check_against_golden(npz, [O.mode_14_outputs(student_sds, img, poses[p]) for p in range(2)], 2e-4)
        npz = numpy.load(os.path.join(golden_dir, 'student_lambda00.npz'))
        img = image_io.load_rgba_png(os.path.join(golden_dir, 'data', 'lambda_00.png'))
        _check_against_golden(npz, [O.mode_14_outputs(lambda00_sds, img, poses[p]) for p in range(2)], 2e-4)


def test_mode_12_is_prefix_of_mode_07(teacher_sds):
    img = synth.synthetic_image(0, 1)[0]
    pose = synth.random_poses(1)[0]
    with torch.no_grad():
        m12 = O.mode_12_outputs(teacher_sds, img, pose)
        dec = O.eyebrow_decomposer(teacher_sds['eyebrow_decomposer'], img.unsqueeze(0)[:, :, 64:192, 192:320])
    assert len(m12) == 22                     # mode_12.py:88-94 returns 22 although it declares 18 (:201)
    for a, b in zip(m12[16:], dec):
        assert torch.equal(a, b)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


@pytest.mark.parametrize('size', [128, 192, 256, 512])
def test_c_oracle_base_grid_within_one_ulp_of_torch(oracle_clib, size):
    out = torch.empty(size)
    oracle_clib.tha4o_base_grid(size, _p(out))
    ref = O.base_grid(1, size, size)[0, 0, :, 0]
    # torch's own linspace differs by 1 ulp between its scalar / AVX2 / AVX-512 / CUDA kernels, so the contract is
    # "the documented scalar formula", checked to 1 ulp of whatever torch build runs here.
    assert (out - ref).abs().max().item() <= 6e-8 * 1.01


@pytest.mark.parametrize('size,amp', [(128, 0.05), (192, 0.3), (256, 1.5), (512, 0.02)])
def test_c_oracle_grid_sample_matches_torch(oracle_clib, size, amp):
    g = torch.Generator().manual_seed(size)
    n, c = 2, 4
    img = synth.synthetic_image(size, n)[:, :, :size, :size].contiguous()
    gc = (torch.randn(n, 2, size, size, generator=g) * amp).contiguous()
    ref = O.apply_grid_change(gc, img)
    out = torch.empty_like(img)
    x0 = torch.empty(n, size, size, dtype=torch.int32)
    y0 = torch.empty_like(x0)
    oracle_clib.tha4o_grid_sample(_p(img), _p(gc), n, c, size, size, _p(out), _p(x0), _p(y0), None, None)
    assert (out - ref).abs().max().item() < 2e-5
    assert x0.min() >= 0 and x0.max() <= size - 1 and y0.min() >= 0 and y0.max() <= size - 1


def test_c_oracle_grid_sample_edge_cases(oracle_clib):
    """Zero offsets reproduce the image; offsets far outside clamp to the border (padding_mode='border')."""
    size, n, c = 128, 1, 4
    img = synth.synthetic_image(7, n)[:, :, :size, :size].contiguous()
    out = torch.empty_like(img)
    gc = torch.zeros(n, 2, size, size)
    oracle_clib.tha4o_grid_sample(_p(img), _p(gc), n, c, size, size, _p(out), None, None, None, None)
    assert (out - img).abs().max().item() < 1e-5
    gc = torch.full((n, 2, size, size), 5.0)
    oracle_clib.tha4o_grid_sample(_p(img), _p(gc), n, c, size, size, _p(out), None, None, None, None)
    assert torch.equal(out, img[:, :, -1:, -1:].expand_as(out).contiguous())
    gc = torch.full((n, 2, size, size), -5.0)
    oracle_clib.tha4o_grid_sample(_p(img), _p(gc), n, c, size, size, _p(out), None, None, None, None)
    assert torch.equal(out, img[:, :, :1, :1].expand_as(out).contiguous())


@pytest.mark.parametrize('hi,ho', [(512, 256), (256, 512), (128, 256)])
def test_c_oracle_resize_matches_torch(oracle_clib, hi, ho):
    a = torch.rand(1, 3, hi, hi, generator=torch.Generator().manual_seed(hi))
    ref = F.interpolate(a, size=(ho, ho), mode='bilinear', align_corners=False)
    out = torch.empty_like(ref)
    oracle_clib.tha4o_resize_bilinear(_p(a), 1, 3, hi, hi, ho, ho, _p(out))
    assert (out - ref).abs().max().item() < 3e-7


def _layout(sd):
    return '\n'.join('%s %s' % (k, list(v.shape)) for k, v in sd.items())


def test_oracle_equals_reference_fixture(golden_dir, teacher_sds, student_sds):
    """tests/golden/reference_posers.npz holds the reference's own state_dict layouts and its mode_07 / mode_12 / mode_14
    outputs on these inputs (a spread-out sample of every tensor, the mean of every 32x32 tile, and mean / mean|x| /
    max|x| of the whole tensor)."""
    npz = numpy.load(os.path.join(golden_dir, 'reference_posers.npz'))
    for grp, sds in (('teacher', teacher_sds), ('student', student_sds)):
        names = sorted(k[len('layout_%s_' % grp):] for k in npz.files if k.startswith('layout_%s_' % grp))
        assert names == sorted(sds)
        for name in names:
            assert _layout(sds[name]) == str(npz['layout_%s_%s' % (grp, name)]), (grp, name)
    img, pose = poser_inputs()
    with torch.no_grad():
        for mode, sds in (('mode_07', teacher_sds), ('mode_12', teacher_sds), ('mode_14', student_sds)):
            mine = getattr(O, mode + '_outputs')(sds, img, pose)
            assert len(mine) == int(npz['%s_count' % mode])
            for i, b in enumerate(mine):
                key = '%s_o%02d' % (mode, i)
                assert list(b.shape) == npz[key + '_shape'].tolist(), key
                assert numpy.abs(spread(b, 256).numpy() - npz[key]).max() <= 1e-6, key
                assert numpy.abs(stats(b) - npz[key + '_stats']).max() <= 1e-6, key
                assert numpy.abs(tile_means(b).astype(numpy.float64) - npz[key + '_tiles']).max() <= 1e-6, key


# ------------------------------------------------------------------------------------------ distillation steps (a16-a18)
def _distill_oracle_results(lambda00_sds):
    from oracle import distill_oracle, make_golden_distill as M
    body_in, face_in = M.distill_inputs()
    res = {}
    sd = lambda00_sds['body_morpher']
    losses, grad = distill_oracle.body_losses_and_grads(sd, body_in['image'], body_in['pose'], body_in['t_posed'], body_in['t_warped'],
                                                        body_in['t_grid'], M.BODY_WEIGHTS)
    p0 = torch.cat([v.reshape(-1) for v in sd.values()])
    res['body'] = dict(weighted=[w * l for w, l in zip(M.BODY_WEIGHTS, losses)], grad=grad,
                       after=distill_oracle.adam_reference(p0, [grad], M.LR))
    sd = lambda00_sds['face_morpher']
    from tha4_b200.distill import face_groundtruth_crop, FACE_LOSS_WEIGHTS
    losses, grad = distill_oracle.face_losses_and_grads(sd, face_in['pose'], face_groundtruth_crop(face_in['posed_face']), face_in['mask'],
                                                        FACE_LOSS_WEIGHTS)
    p0 = torch.cat([v.reshape(-1) for v in sd.values()])
    res['face'] = dict(weighted=[w * l for w, l in zip(FACE_LOSS_WEIGHTS, losses)], grad=grad,
                       after=distill_oracle.adam_reference(p0, [grad], M.LR))
    return res


def test_distill_oracle_matches_reference_training_iteration_golden(golden_dir, lambda00_sds):
    """tests/golden/distill_lambda00.npz was written by oracle/make_golden_distill.py from the reference's OWN
    run_training_iteration (real protocols, SumLoss, Adam; stub teacher returning fixed tensors).  The restated step must
    reproduce its weighted loss terms, gradient and post-Adam parameters."""
    from oracle import make_golden_distill as M
    npz = numpy.load(os.path.join(golden_dir, 'distill_lambda00.npz'))
    res = _distill_oracle_results(lambda00_sds)
    names = {'body': ['full_blended_loss', 'full_warped_loss', 'full_grid_change_loss', 'full_color_change_loss'],
             'face': ['full_loss', 'eye_mouth_loss']}
    for net in ('body', 'face'):
        for name, val in zip(names[net], res[net]['weighted']):
            ref = float(npz['%s_log_%s' % (net, name)])
            assert abs(val - ref) <= 2e-6 * max(1.0, abs(ref)), (net, name, val, ref)
        assert abs(sum(res[net]['weighted']) - float(npz['%s_log_loss' % net])) <= 5e-6
        g = res[net]['grad']
        stats = npz['%s_grad_stats' % net]
        assert g.numel() == int(stats[3])
        gsub = torch.from_numpy(npz['%s_grad_sub' % net])
        assert (g[::M.GRAD_STRIDE] - gsub).abs().max().item() <= 1e-5 * max(1.0, float(stats[2])), net
        assert abs(g.double().norm().item() - stats[0]) <= 1e-4 * stats[0], net
        after = torch.from_numpy(npz['%s_params_after_sub' % net])
        assert (res[net]['after'][::M.GRAD_STRIDE] - after).abs().max().item() <= 2e-7, net


def test_distill_oracle_equals_reference_iteration_fixture(golden_dir, lambda00_sds):
    """tests/golden/reference_distill.npz: the gradient and post-Adam parameters of the reference's own training
    iteration (oracle/make_golden_pins.py), sampled on a different grid than distill_lambda00.npz."""
    npz = numpy.load(os.path.join(golden_dir, 'reference_distill.npz'))
    res = _distill_oracle_results(lambda00_sds)
    for net in ('body', 'face'):
        g = res[net]['grad']
        assert g.numel() == int(npz['%s_numel' % net])
        gl = torch.from_numpy(npz['%s_grad_sub' % net])
        assert (spread(g, gl.numel()) - gl).abs().max().item() <= 1e-5 * max(1.0, float(npz['%s_grad_absmax' % net])), net
        after = torch.from_numpy(npz['%s_params_after_sub' % net])
        assert (spread(res[net]['after'], after.numel()) - after).abs().max().item() <= 2e-7, net
        assert abs(sum(res[net]['weighted']) - float(npz['%s_logged_loss' % net])) <= 5e-6, net


# ------------------------------------------------------------------------------------------ image I/O on either side of the path
def test_image_loader_and_output_conversion_equal_reference(golden_dir):
    """PNG -> poser tensor (full_manual_poser.py:329-339 via extract_pytorch_image_from_filelike) and poser output -> uint8
    sRGB RGBA (convert_output_image_from_torch_to_numpy, src/tha4/image_util.py:41-58) against what the reference's
    functions returned (tests/golden/reference_image_io.npz)."""
    from tha4_b200 import image_util
    npz = numpy.load(os.path.join(golden_dir, 'reference_image_io.npz'))
    png = os.path.join(golden_dir, 'data', 'lambda_00.png')
    ours, orc = image_util.load_poser_image(png), image_io.load_rgba_png(png)
    assert list(ours.shape) == list(orc.shape) == npz['loaded_shape'].tolist() == [4, 512, 512]
    for t in (ours, orc):
        assert numpy.abs(spread(t, 8192).numpy() - npz['loaded_sub']).max() <= 1e-6
        assert numpy.abs(stats(t) - npz['loaded_stats']).max() <= 1e-6
    out = synth.synthetic_image(3, 1)[0]
    a = image_util.poser_output_to_rgba_uint8(out)
    assert list(a.shape) == npz['output_rgba8_shape'].tolist() == [512, 512, 4] and a.dtype == npz['output_rgba8_sub'].dtype == numpy.uint8
    a = spread(torch.from_numpy(a), 8192).numpy()
    assert numpy.abs(a.astype(int) - npz['output_rgba8_sub'].astype(int)).max() <= 1        # uint8 rounding of float32 vs float64 pow


def test_image_loader_golden_statistics(golden_dir):
    """Same pin for the GPU box (no reference there): statistics of the loaded lambda_00 image recorded from the reference's
    loader when the fixture was generated."""
    from tha4_b200 import image_util
    img = image_util.load_poser_image(os.path.join(golden_dir, 'data', 'lambda_00.png')).double()
    stats = numpy.load(os.path.join(golden_dir, 'image_lambda00_stats.npz'))['stats']
    got = numpy.array([img.mean().item(), img.abs().mean().item(), img[3].mean().item(), img[:3, 200:300, 200:300].mean().item()])
    assert numpy.abs(got - stats).max() <= 1e-7


# ------------------------------------------------------------------------------------------ poser API surface (a1, a2)
def test_pose_schema_and_poser_surface_equal_reference(golden_dir):
    """Every pose parameter group (name, arity, category, default, range, discreteness -- pose_parameters.py:4-35) and the
    poser getters the GUIs call (poser.py:132-161) match the reference objects field by field, as recorded in
    tests/golden/reference_pins.json."""
    from tha4_b200.poser.modes.pose_parameters import get_pose_parameters as our_get
    ref = json.load(open(os.path.join(golden_dir, 'reference_pins.json')))['pose']
    ours = our_get()
    assert ours.get_parameter_count() == ref['parameter_count'] == 45
    og = ours.get_pose_parameter_groups()
    assert len(og) == len(ref['groups'])
    for a, b in zip(og, ref['groups']):
        assert a.get_group_name() == b['group_name'] and a.get_arity() == b['arity']
        assert a.get_parameter_index() == b['parameter_index'] and a.get_parameter_names() == b['parameter_names']
        assert [a.get_category().name, a.get_category().value] == b['category']
        assert a.get_default_value() == b['default_value'] and tuple(a.get_range()) == tuple(b['range'])
        assert a.is_discrete() == b['discrete']
    for i in range(45):
        assert ours.get_parameter_name(i) == ref['parameter_names'][i]
        assert ours.get_parameter_index(ref['parameter_names'][i]) == i
    ssd = synth.student_state_dicts(0)
    from tha4_b200.poser.modes import mode_14
    oposer = mode_14.create_poser(torch.device('cuda:0'), state_dicts=ssd)          # construction needs no GPU (lazy modules)
    rposer = ref['mode_14_poser']
    assert oposer.get_image_size() == rposer['image_size'] and oposer.get_output_length() == rposer['output_length']
    assert oposer.get_num_parameters() == rposer['num_parameters'] and str(oposer.get_dtype()) == rposer['dtype']


def test_display_conversion_pinned_to_reference_functions(golden_dir):
    """oracle/image_io.frame_to_srgb8 restates the puppeteers' post-processing (a wx app that cannot be imported here);
    its building blocks are the reference's own convert_linear_to_srgb / torch_linear_to_srgb, whose results on this
    input are recorded in tests/golden/reference_image_io.npz."""
    npz = numpy.load(os.path.join(golden_dir, 'reference_image_io.npz'))
    x = display_input()
    o = torch.clip((x + 1.0) / 2.0, 0.0, 1.0)
    srgb = torch.cat([image_io.linear_to_srgb_torch(o[0:3]), o[3:4]], dim=0)
    assert numpy.array_equal(spread(srgb, 8192).numpy(), npz['display_srgb_sub'])
    assert numpy.abs(stats(srgb) - npz['display_srgb_stats']).max() <= 1e-9
    plain = image_io.frame_to_srgb8(x, 0)
    assert numpy.array_equal(spread(plain, 8192).numpy(), npz['display_srgb8_sub'])
    white = image_io.frame_to_srgb8(x, 4)
    assert (white[:, :, 3] == 255).all()
