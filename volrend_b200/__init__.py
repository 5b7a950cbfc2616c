"""volrend_b200 -- B200-native PlenOctree ray-marcher behind volrend's renderer surface.

The product is ``libvolrend_b200.so`` (hand-written sm_100a kernels + the C-ABI in
``include/volrend_b200.h``).  This package is the thin host-side mirror of the reference's
``N3Tree`` / ``Camera`` / ``RenderOptions`` / ``VolumeRenderer`` / ``launch_renderer`` plus
synthetic-scene generators; see DESIGN.md.
"""
from .host import (CAMERA_DEFAULT_FOCAL_LENGTH, VOLREND_GLOBAL_BASIS_MAX, Camera, DataFormat, N3Tree,
                   RenderOptions, VolumeRenderer, MultiGpuRenderer, VR_MG_TILES, VR_MG_VIEWS, launch_renderer, render_bands, render_bands_batch, render_batch, render_rays, camera_rays, render_frames_host, render_frames_png, write_png_file)
from ._capi import LIB_PATH, VolrendError, lib

__all__ = ["N3Tree", "Camera", "RenderOptions", "VolumeRenderer", "DataFormat", "launch_renderer", "MultiGpuRenderer", "VR_MG_VIEWS", "VR_MG_TILES",
           "render_batch", "render_rays", "camera_rays", "render_bands", "render_bands_batch", "render_frames_host", "render_frames_png", "write_png_file", "lib", "LIB_PATH", "VolrendError",
           "CAMERA_DEFAULT_FOCAL_LENGTH", "VOLREND_GLOBAL_BASIS_MAX"]
