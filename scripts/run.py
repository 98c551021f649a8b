#!/usr/bin/env python
"""CLI with the option surface of the reference's scripts/run.py (same flags, defaults, stage order, exit codes;
scripts/run.py:58-155, 253-256, 272-302, 311-338), driving the B200 engine.  `--weights` takes an
ultralytics YOLOv8 detection checkpoint (read without the ultralytics package) or a caesar_yolo_b200 weight file
(caesar_yolo_b200/weights.py).  Multi-GPU: launch with torchrun (one rank per GPU)
instead of mpirun; `--devices` defaults to cuda:0 here because this build has no CPU path."""
import argparse
import logging
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

logging.basicConfig(format="%(asctime)-15s %(levelname)s - %(message)s")
logger = logging.getLogger("caesar_yolo_b200")
logger.setLevel(logging.INFO)


def parse_args(argv=None):
    p = argparse.ArgumentParser(description='CAESAR-YOLO options')
    p.add_argument('--image', required=False, type=str)
    p.add_argument('--datalist', required=False)
    p.add_argument('--maxnimgs', required=False, type=int, default=-1)
    p.add_argument('--weights', required=True)
    p.add_argument('--imgsize', dest='imgsize', required=False, type=int, default=640)
    p.add_argument('--preprocessing', dest='preprocessing', action='store_true')
    p.add_argument('--normalize_minmax', dest='normalize_minmax', action='store_true')
    p.add_argument('-norm_min', '--norm_min', dest='norm_min', type=float, default=0.)
    p.add_argument('-norm_max', '--norm_max', dest='norm_max', type=float, default=1.)
    p.add_argument('--subtract_bkg', dest='subtract_bkg', action='store_true')
    p.add_argument('-sigma_bkg', '--sigma_bkg', dest='sigma_bkg', type=float, default=3)
    p.add_argument('--use_box_mask_in_bkg', dest='use_box_mask_in_bkg', action='store_true')
    p.add_argument('-bkg_box_mask_fract', '--bkg_box_mask_fract', dest='bkg_box_mask_fract', type=float, default=0.7)
    p.add_argument('-bkg_chid', '--bkg_chid', dest='bkg_chid', type=int, default=-1)
    p.add_argument('--clip_shift_data', dest='clip_shift_data', action='store_true')
    p.add_argument('-sigma_clip', '--sigma_clip', dest='sigma_clip', type=float, default=1)
    p.add_argument('--clip_data', dest='clip_data', action='store_true')
    p.add_argument('-sigma_clip_low', '--sigma_clip_low', dest='sigma_clip_low', type=float, default=10)
    p.add_argument('-sigma_clip_up', '--sigma_clip_up', dest='sigma_clip_up', type=float, default=10)
    p.add_argument('-clip_chid', '--clip_chid', dest='clip_chid', type=int, default=-1)
    p.add_argument('--zscale_stretch', dest='zscale_stretch', action='store_true')
    p.add_argument('--zscale_contrasts', dest='zscale_contrasts', type=str, default='0.25,0.25,0.25')
    p.add_argument('--chan3_preproc', dest='chan3_preproc', action='store_true')
    p.add_argument('-sigma_clip_baseline', '--sigma_clip_baseline', dest='sigma_clip_baseline', type=float, default=0)
    p.add_argument('-nchannels', '--nchannels', dest='nchannels', type=int, default=1)
    p.add_argument('--scoreThr', default=0.7, type=float)
    p.add_argument('--iouThr', default=0.5, type=float)
    p.add_argument('--merge_overlap_iou_thr_soft', default=0.3, type=float)
    p.add_argument('--merge_overlap_iou_thr_hard', default=0.8, type=float)
    p.add_argument('--xmin', dest='xmin', type=int, default=-1)
    p.add_argument('--xmax', dest='xmax', type=int, default=-1)
    p.add_argument('--ymin', dest='ymin', type=int, default=-1)
    p.add_argument('--ymax', dest='ymax', type=int, default=-1)
    p.add_argument('--split_img_in_tiles', dest='split_img_in_tiles', action='store_true')
    p.add_argument('--tile_xsize', dest='tile_xsize', type=int, default=512)
    p.add_argument('--tile_ysize', dest='tile_ysize', type=int, default=512)
    p.add_argument('--tile_xstep', dest='tile_xstep', type=float, default=1.0)
    p.add_argument('--tile_ystep', dest='tile_ystep', type=float, default=1.0)
    p.add_argument('--max_ntasks_per_worker', dest='max_ntasks_per_worker', type=int, default=100)
    p.add_argument('--devices', required=False, type=str, default="cuda:0")
    p.add_argument('--multigpu', dest='multigpu', action='store_true')
    p.add_argument('--draw_plots', dest='draw_plots', action='store_true')
    p.add_argument('--draw_class_label_in_caption', dest='draw_class_label_in_caption', action='store_true')
    p.add_argument('--save_plots', dest='save_plots', action='store_true')
    p.add_argument('--save_tile_catalog', dest='save_tile_catalog', action='store_true')
    p.add_argument('--save_tile_region', dest='save_tile_region', action='store_true')
    p.add_argument('--save_tile_img', dest='save_tile_img', action='store_true')
    p.add_argument('--precision', required=False, type=str, default=None, choices=['fp16', 'bf16'],
                   help='B200 build only: 16-bit storage of weights/activations (default fp16; same tensor-core rate)')
    p.add_argument('--measure_sources', dest='measure_sources', action='store_true',
                   help='B200 build only: add peak, flux density, centroid, shape and sky position to every catalog source')
    p.add_argument('--measure_noise', dest='measure_noise', action='store_true',
                   help='B200 build only: add local background, rms, S/N, background-subtracted flux density and its '
                        'error to every catalog source (implies --measure_sources)')
    p.add_argument('--noise_frame', dest='noise_frame', type=int, default=16,
                   help='B200 build only: width in pixels of the frame around each box that --measure_noise clips')
    p.add_argument('--save_bkg_maps', dest='save_bkg_maps', action='store_true',
                   help='B200 build only: write the background and rms maps of a FITS image (bkgmap_<id>.fits, '
                        'rmsmap_<id>.fits)')
    p.add_argument('--save_snr_maps', dest='save_snr_maps', action='store_true',
                   help='B200 build only: also write the background-subtracted and S/N maps of a FITS image '
                        '(resmap_<id>.fits, snrmap_<id>.fits; implies --save_bkg_maps)')
    p.add_argument('--bkg_box', dest='bkg_box', type=int, default=101,
                   help='B200 build only: side in pixels (odd, >= 3) of the box each --save_bkg_maps node clips')
    p.add_argument('--bkg_grid', dest='bkg_grid', type=int, default=25,
                   help='B200 build only: step in pixels (>= 1) of the --save_bkg_maps node lattice')
    p.add_argument('--bkg_mask_sources', dest='bkg_mask_sources', action='store_true',
                   help='B200 build only: mask the catalog boxes out of the --measure_noise frames and the '
                        '--save_bkg_maps node boxes, and fill the map nodes left without pixels from their neighbours')
    p.add_argument('--bkg_estimator', dest='bkg_estimator', type=str, default='mean', choices=['mean', 'median'],
                   help='B200 build only: centre of the --measure_noise and --save_bkg_maps sigma clipping (median: '
                        "astropy's sigma_clipped_stats default; bkg is the clipped median)")
    p.add_argument('--detect_outfile', required=False, type=str, default="")
    p.add_argument('--detect_outfile_json', required=False, type=str, default="")
    args = p.parse_args(argv)
    args.measure_sources = args.measure_sources or args.measure_noise   # S/N and flux_bkgsub need the peak and sum
    args.save_bkg_maps = args.save_bkg_maps or args.save_snr_maps       # res / snr are made from the bkg / rms nodes
    return args


def validate_args(args):
    """scripts/run.py:158-190."""
    if not (args.image and args.image != ""):
        logger.error("Argument --image is required for detect task!")
        return -1
    if not os.path.isfile(args.image):
        logger.error("Image argument must be an existing image on filesystem!")
        return -1
    if not args.image.endswith(('.fits', '.png', '.jpg')):
        logger.error("Image must have .fits/.png/.jpg extension!")
        return -1
    if not args.image.endswith('.fits') and args.split_img_in_tiles:
        logger.error("Tiled runs need a FITS image (the reference reads tiles with read_fits_crop only)")
        return -1
    if args.maxnimgs == 0 or (args.maxnimgs < 0 and args.maxnimgs != -1):
        logger.error("Invalid maxnimgs given (hint: give -1 or >0)!")
        return -1
    if args.weights == "" or not os.path.isfile(args.weights):
        logger.error("Given weight file %s not existing or not a file!" % args.weights)
        return -1
    if args.noise_frame < 1:
        logger.error("Invalid noise_frame given (hint: give a frame width >= 1 pixel)!")
        return -1
    if args.bkg_box < 3 or args.bkg_box % 2 == 0:
        logger.error("Invalid bkg_box given (hint: give an odd box side >= 3 pixels)!")
        return -1
    if args.bkg_grid < 1:
        logger.error("Invalid bkg_grid given (hint: give a grid step >= 1 pixel)!")
        return -1
    if args.bkg_estimator not in ('mean', 'median'):
        logger.error("Invalid bkg_estimator given (hint: give mean or median)!")
        return -1
    return 0


def build_stages(args):
    """Stage list in the reference's fixed order (scripts/run.py:272-293)."""
    from caesar_yolo_b200.preprocessing import (BkgSubtractor, SigmaClipShifter, SigmaClipper, ChanResizer,
                                                ZScaleTransformer, Chan3Trasformer, MinMaxNormalizer)
    zc = [float(x) for x in args.zscale_contrasts.split(',')]
    st = []
    if args.subtract_bkg:
        st.append(BkgSubtractor(sigma=args.sigma_bkg, use_mask_box=args.use_box_mask_in_bkg,
                                mask_fract=args.bkg_box_mask_fract, chid=args.bkg_chid))
    if args.clip_shift_data:
        st.append(SigmaClipShifter(sigma=args.sigma_clip, chid=args.clip_chid))
    if args.clip_data:
        st.append(SigmaClipper(sigma_low=args.sigma_clip_low, sigma_up=args.sigma_clip_up, chid=args.clip_chid))
    if args.nchannels > 1:
        st.append(ChanResizer(nchans=args.nchannels))
    if args.zscale_stretch:
        st.append(ZScaleTransformer(contrasts=zc))
    if args.chan3_preproc:
        st.append(Chan3Trasformer(sigma_clip_baseline=args.sigma_clip_baseline, sigma_clip_low=args.sigma_clip_low,
                                  sigma_clip_up=args.sigma_clip_up, zscale_contrast=zc[0]))
    if args.normalize_minmax:
        st.append(MinMaxNormalizer(norm_min=args.norm_min, norm_max=args.norm_max))
    return st


def main(argv=None):
    try:
        args = parse_args(argv)
    except SystemExit:
        return 1
    if validate_args(args) < 0:
        return 1
    if args.chan3_preproc and args.nchannels != 3:
        logger.error("You selected chan3_preproc pre-processing options, you must set nchannels options to 3!")
        return 1
    devices = [str(x) for x in args.devices.split(',')]
    if not devices:
        return 1
    import torch
    import torch.distributed as dist
    if int(os.environ.get('WORLD_SIZE', '1')) > 1 and not dist.is_initialized():
        torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
        dist.init_process_group('nccl')
    from caesar_yolo_b200.config import CONFIG
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    from caesar_yolo_b200.preprocessing import DataPreprocessor
    stages = build_stages(args)
    dp = None
    if args.preprocessing:
        if not stages:
            logger.warning("No pre-processing steps defined ...")
        else:
            dp = DataPreprocessor(stages)
    CONFIG.update({
        'img_size': args.imgsize, 'preprocess_fcn': dp, 'image_path': args.image, 'image_xmin': args.xmin,
        'image_xmax': args.xmax, 'image_ymin': args.ymin, 'image_ymax': args.ymax, 'mpi': None,
        'split_image_in_tiles': args.split_img_in_tiles, 'tile_xsize': args.tile_xsize, 'tile_ysize': args.tile_ysize,
        'tile_xstep': args.tile_xstep, 'tile_ystep': args.tile_ystep,
        'max_ntasks_per_worker': args.max_ntasks_per_worker, 'devices': devices, 'use_multi_gpu': args.multigpu,
        'iou_thr': args.iouThr, 'score_thr': args.scoreThr,
        'merge_overlap_iou_thr_soft': args.merge_overlap_iou_thr_soft,
        'merge_overlap_iou_thr_hard': args.merge_overlap_iou_thr_hard, 'outfile': args.detect_outfile,
        'outfile_json': args.detect_outfile_json, 'draw_plot': args.draw_plots,
        'draw_class_label_in_caption': args.draw_class_label_in_caption, 'save_plot': args.save_plots,
        'save_tile_catalog': args.save_tile_catalog, 'save_tile_region': args.save_tile_region,
        'save_tile_img': args.save_tile_img, 'precision': args.precision, 'measure_sources': args.measure_sources,
        'measure_noise': args.measure_noise, 'noise_frame': args.noise_frame, 'save_bkg_maps': args.save_bkg_maps,
        'bkg_box': args.bkg_box, 'bkg_grid': args.bkg_grid, 'bkg_mask_sources': args.bkg_mask_sources,
        'bkg_estimator': args.bkg_estimator, 'save_snr_maps': args.save_snr_maps,
    })
    model = YOLO(args.weights, precision=args.precision)
    sfinder = SFinder(model, CONFIG)
    status = sfinder.run_parallel() if args.split_img_in_tiles else sfinder.run()
    if status < 0:
        logger.error("sfinder run failed, see logs...")
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
