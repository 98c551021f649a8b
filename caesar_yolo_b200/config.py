"""Defaults dictionary with the reference's keys and values (caesar_yolo/config.py:4-59).  `scripts/run.py` mutates it
in place exactly like the reference does (scripts/run.py:311-338)."""

CONFIG = {
    # - Image resize
    'img_size': 640,
    # - Preprocessor function
    'preprocess_fcn': None,
    # - Image read options
    'image_path': '',
    'image_xmin': 0,
    'image_xmax': 0,
    'image_ymin': 0,
    'image_ymax': 0,
    # - Image parallel read options ('mpi' is accepted for compatibility; ranks come from torch.distributed)
    'mpi': None,
    'split_image_in_tiles': False,
    'tile_xsize': 256,
    'tile_ysize': 256,
    'tile_xstep': 1.0,
    'tile_ystep': 1.0,
    'max_ntasks_per_worker': 100,
    # - Source detection options
    'devices': ['cpu'],
    'use_multi_gpu': False,
    'iou_thr': 0.5,
    'merge_overlap_iou_thr_soft': 0.3,
    'merge_overlap_iou_thr_hard': 0.8,
    'score_thr': 0.7,
    # - Catalog json output options
    'save_catalog': True,
    'save_tile_catalog': False,
    'outfile_json': '',
    # - DS9 region output options
    'save_region': True,
    'save_tile_region': False,
    'outfile': '',
    # - Image output file options
    'save_img': False,
    'save_tile_img': False,
    # - Save inference plot
    'draw_plot': False,
    'draw_class_label_in_caption': True,
    'save_plot': False,
    # - Per-source measurements (not in the reference): peak, flux density, centroid, shape, sky position
    'measure_sources': False,
    # - Local background, noise and S/N of every source (not in the reference; implies measure_sources): sigma-clipped
    #   mean / std of a frame of noise_frame pixels around each box
    'measure_noise': False,
    'noise_frame': 16,
    # - Background and rms maps of the image (not in the reference; FITS input): the statistic of measure_noise over
    #   boxes of bkg_box pixels on a lattice of step bkg_grid, interpolated bilinearly; bkgmap_<id>.fits, rmsmap_<id>.fits
    'save_bkg_maps': False,
    'bkg_box': 101,
    'bkg_grid': 25,
    # - Background-subtracted and S/N maps of the image (not in the reference; FITS input; implies save_bkg_maps):
    #   (image - bkg) and (image - bkg) / rms at every pixel of the bkg / rms maps; resmap_<id>.fits, snrmap_<id>.fits
    'save_snr_maps': False,
    # - Mask the catalog boxes out of the measure_noise frames and the save_bkg_maps node boxes (not in the reference);
    #   map nodes left without pixels are filled from their neighbours.  Alone it changes nothing (one warning)
    'bkg_mask_sources': False,
    # - Centre of the sigma clipping of measure_noise and save_bkg_maps (not in the reference): 'mean' or 'median'
    #   (astropy's sigma_clipped_stats default; bkg is then the clipped median).  Alone it changes nothing (one warning)
    'bkg_estimator': 'mean',
    # - Catalog completeness by injection and recovery (not in the reference; FITS input): inject_sources beam-shaped
    #   point sources per round at empty positions, with S/N log-uniform in inject_snr_range against the rms map of the
    #   save_bkg_maps options, detected again; inject_<id>.json.  0: off
    'inject_sources': 0,
    'inject_rounds': 1,
    'inject_snr_range': (3.0, 100.0),
    'inject_seed': 0,
    # - Catalog reliability from the inverted image (not in the reference; FITS input): the catalog of -I, the peak S/N
    #   of both catalogs against the S/N map of the save_bkg_maps options, tables over inject_snr_range and the score;
    #   reliability_<id>.json (and .reg with save_region)
    'reliability': False,
}
