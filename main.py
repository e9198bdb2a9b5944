"""CLI of the B200-native video-feature engine: the flags of the reference's main.py (main.py:93-149), same names,
defaults and choices.  ``--device_ids`` starts one process per GPU (reference: one thread per GPU); ``--cpu`` is
refused -- the reference's CPU path is what ``bench.py --impl reference`` times, the engine itself has no CPU path.
"""
import argparse
import functools

import numpy  # noqa: F401  (kept first, as in the reference)
import torch  # noqa: F401

from video_features_b200.utils import form_list_from_user_input, sanity_check

SUPPORTED = ['i3d', 'raft', 'CLIP-ViT-B/32', 'CLIP-ViT-B/16', 'CLIP4CLIP-ViT-B-32', 'resnet18', 'resnet34', 'resnet50',
             'resnet101', 'resnet152']


def build_extractor(args):
    """feature_type -> extractor (main.py:15-41)."""
    if args.feature_type in ['CLIP-ViT-B/32', 'CLIP-ViT-B/16', 'CLIP4CLIP-ViT-B-32']:
        from video_features_b200.extract.extract_clip import ExtractCLIP
        return ExtractCLIP(args)
    if args.feature_type == 'i3d':
        from video_features_b200.extract.extract_i3d import ExtractI3D
        return ExtractI3D(args)
    if args.feature_type == 'raft':
        from video_features_b200.extract.extract_raft import ExtractRAFT
        return ExtractRAFT(args)
    if args.feature_type in ['resnet18', 'resnet34', 'resnet50', 'resnet101', 'resnet152']:
        from video_features_b200.extract.extract_resnet import ExtractResNet
        return ExtractResNet(args)
    if args.feature_type in ['vggish', 'r21d_rgb', 'pwc', 'vggish_torch']:
        raise NotImplementedError(f'{args.feature_type}: outside the hot path this engine rebuilds (SURVEY.md §2)')
    raise NotADirectoryError                      # main.py:41


def _pin_path_list(args):
    """Resolve the user's listing ONCE, here in the parent: every worker then sees the same list in the same order (a
    directory glob is unordered, and shard r is only meaningful against one enumeration).  Returns the list."""
    paths = form_list_from_user_input(args)
    if paths and isinstance(paths[0], tuple):
        args.video_paths, args.flow_paths = [p[0] for p in paths], [p[1] for p in paths]
    else:
        args.video_paths, args.flow_paths = list(paths), None
    args.file_with_video_paths = args.video_dir = args.flow_dir = None
    return paths


def _save_gathered(target, blocks):
    """--gather_features: every video's feature block, list order, in one .npz (rows + per-video row counts)."""
    import numpy as np
    rows = np.concatenate([b.numpy() for b in blocks]) if blocks else np.zeros((0, 0), np.float32)
    np.savez(target, features=rows, rows_per_video=np.array([b.shape[0] for b in blocks], dtype=np.int64))
    print(f'gathered {len(blocks)} feature blocks ({rows.shape[0]} rows) -> {target}')


def parallel_feature_extraction(args):
    from video_features_b200.dispatch import parallel_feature_extraction as run
    video_paths = _pin_path_list(args)
    gather = getattr(args, 'gather_features', None)
    key = {'i3d': (args.streams or ['rgb'])[0]}.get(args.feature_type, args.feature_type)
    run(functools.partial(build_extractor, args), len(video_paths), args.device_ids,
        gather_key=key if gather else None, on_gathered=functools.partial(_save_gathered, gather) if gather else None)


_FEATURE_TYPES = ('i3d vggish r21d_rgb resnet18 resnet34 resnet50 resnet101 resnet152 raft pwc CLIP-ViT-B/32 CLIP-ViT-B/16 '
                  'CLIP4CLIP-ViT-B-32 vggish_torch').split()

# (flag, argparse keywords): names, types, defaults, choices and dests are the reference's (main.py:93-149)
_FLAGS = [
    ('--feature_type', dict(required=True, choices=_FEATURE_TYPES, help='which extractor to run')),
    ('--video_paths', dict(nargs='+', help='videos to process')),
    ('--flow_paths', dict(nargs='+', help='folders of precomputed flow images, one per video (I3D --flow_type flow)')),
    ('--file_with_video_paths', dict(help='text file, one video path per line')),
    ('--video_dir', dict(type=str, help='directory whose files are all processed')),
    ('--flow_dir', dict(type=str, help='root of <video id>/flow_{x,y}_NNNNNN.jpg trees')),
    ('--device_ids', dict(type=int, nargs='+', help='GPUs to use: one process per id')),
    ('--cpu', dict(action='store_true', help='accepted for compatibility; refused at run time')),
    ('--tmp_path', dict(default='./tmp', help='scratch folder')),
    ('--keep_tmp_files', dict(dest='keep_tmp_files', action='store_true', default=False, help='keep the scratch files')),
    ('--on_extraction', dict(default='print', choices=['print', 'save_numpy', 'save_pickle'], help='sink of the features')),
    ('--output_path', dict(default='./output', help='root of the saved features')),
    ('--output_direct', dict(action='store_true', help='save as <output_path>/<video stem>.npy')),
    ('--extraction_fps', dict(type=float, help='resample to this frame rate first (I3D; refused by RAFT and ResNet)')),
    ('--extract_method', dict(type=str, help='frame sampler: uni_N or fix_N')),
    ('--stack_size', dict(type=int, help='frames per I3D stack')),
    ('--step_size', dict(type=int, help='frames between I3D stacks')),
    ('--streams', dict(nargs='+', choices=['flow', 'rgb'], help='I3D streams (default: both)')),
    ('--flow_type', dict(choices=['raft', 'pwc', 'flow'], default='pwc', help='optical flow feeding the I3D flow stream')),
    ('--batch_size', dict(type=int, default=1, help='frame pairs per RAFT call, frames per ResNet call')),
    ('--resize_to_larger_edge', dict(dest='resize_to_smaller_edge', action='store_false', default=True,
                                    help='--side_size applies to the larger edge instead of the smaller one')),
    ('--side_size', dict(type=int, help='RAFT: resize frames to this edge length first')),
    ('--show_pred', dict(dest='show_pred', action='store_true', default=False, help='print class predictions (not built here)')),
    # not in the reference: after extraction, ONE all-gather (NCCL over NVLink) returns every rank's feature blocks and
    # rank 0 writes them, list order, to this .npz
    ('--gather_features', dict(type=str, default=None, help='also all-gather the features of all GPUs into this .npz')),
]


def make_parser():
    parser = argparse.ArgumentParser(description='B200-native video feature extraction')
    for flag, kw in _FLAGS:
        parser.add_argument(flag, **kw)
    return parser


if __name__ == "__main__":
    args = make_parser().parse_args()
    if args.on_extraction != 'print':
        print(f'features -> {args.output_path}')
    if args.keep_tmp_files:
        print(f'scratch files stay in {args.tmp_path}')
    sanity_check(args)
    if args.cpu:
        raise SystemExit('--cpu: this engine has no CPU path (the reference CPU flow is timed by '
                         '`python bench.py --impl reference`); pass --device_ids')
    if not args.device_ids:
        args.device_ids = [0]
    parallel_feature_extraction(args)
