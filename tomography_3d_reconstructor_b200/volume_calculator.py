#!/usr/bin/env python3
"""Drop-in `volume_calculator` module: the reference's VolumeCalculator (volume_calculator.py:10-131).

Voxel counts and index extrema are reduced on the device (warp-shuffle trees over the bit-packed volume); the
float64 scalar arithmetic stays on the host in the reference's exact order, so results are bit-identical.
"""
from __future__ import annotations

import numpy as np

from . import engine


class VolumeCalculator:
    """Handles volume calculations and object property analysis (B200)."""

    def __init__(self):
        pass

    @staticmethod
    def _dv(voxel_data: np.ndarray) -> engine.DeviceVolume:
        """The device volume of a (Z,H,W) occupancy array.  bool arrays are what the pipeline produces; like the reference
        (np.sum / np.where work on any dtype, volume_calculator.py:20,34,40) other numeric dtypes are accepted as long as
        they are occupancies, i.e. hold only 0 and 1 -- then np.sum IS the voxel count the device computes.  Anything else
        (say 0/255 masks, where the reference would return 255 x the volume) is refused rather than silently reinterpreted."""
        if not isinstance(voxel_data, np.ndarray) or voxel_data.ndim != 3:
            raise TypeError("voxel_data must be a numpy array (Z,H,W)")
        if voxel_data.dtype != np.bool_:
            known = engine.volumes.lookup(voxel_data)
            if known is not None:
                return known
            if voxel_data.dtype.kind not in "uif" or not bool(np.logical_or(voxel_data == 0, voxel_data == 1).all()):
                raise TypeError("voxel_data must be a bool array or a numeric array holding only 0 and 1")
        return engine.volume_from_host(voxel_data)

    def calculate_voxel_volume(self, voxel_data: np.ndarray, mm_per_pixel_x: float,
                               mm_per_pixel_y: float, mm_per_slice: float) -> float:
        """Calculate volume from voxel data in mm³ (volume_calculator.py:16-21)."""
        voxel_volume = mm_per_pixel_x * mm_per_pixel_y * mm_per_slice
        total_volume = np.int64(self._dv(voxel_data).slice_counts().sum()) * voxel_volume
        return total_volume

    def calculate_voxel_volume_variable_depth(self, voxel_data: np.ndarray, mm_per_pixel_x: float,
                                              mm_per_pixel_y: float, slice_depths: np.ndarray) -> float:
        """Calculate volume with variable slice depths in mm³ (volume_calculator.py:23-35)."""
        if len(slice_depths) == 0:
            return 0.0

        counts = self._dv(voxel_data).slice_counts()
        total_volume = 0.0
        for z in range(min(voxel_data.shape[0], len(slice_depths))):
            slice_volume = mm_per_pixel_x * mm_per_pixel_y * slice_depths[z]
            total_volume += counts[z] * slice_volume

        return total_volume

    def calculate_bounding_box(self, voxel_data: np.ndarray, mm_per_pixel_x: float,
                               mm_per_pixel_y: float, mm_per_slice: float) -> dict:
        """Calculate bounding box in mm (volume_calculator.py:37-57)."""
        b = self._dv(voxel_data).bbox()
        if b is None:
            raise ValueError("zero-size array to reduction operation minimum which has no identity")
        zmin, zmax, ymin, ymax, xmin, xmax = (np.int64(v) for v in b)

        bbox_x = (xmin * mm_per_pixel_x, xmax * mm_per_pixel_x)
        bbox_y = (ymin * mm_per_pixel_y, ymax * mm_per_pixel_y)
        bbox_z = (zmin * mm_per_slice, zmax * mm_per_slice)

        bbox_dimensions = (bbox_x[1] - bbox_x[0], bbox_y[1] - bbox_y[0], bbox_z[1] - bbox_z[0])

        return {'x': bbox_x, 'y': bbox_y, 'z': bbox_z, 'dimensions': bbox_dimensions}

    def calculate_bounding_box_variable_depth(self, voxel_data: np.ndarray, mm_per_pixel_x: float,
                                              mm_per_pixel_y: float, slice_depths: np.ndarray) -> dict:
        """Calculate bounding box in mm with variable slice depths (volume_calculator.py:59-94)."""
        b = self._dv(voxel_data).bbox()

        if b is None or len(slice_depths) == 0:
            return {'x': (0, 0), 'y': (0, 0), 'z': (0, 0), 'dimensions': (0, 0, 0)}

        zmin, zmax, ymin, ymax, xmin, xmax = (np.int64(v) for v in b)
        bbox_x = (xmin * mm_per_pixel_x, xmax * mm_per_pixel_x)
        bbox_y = (ymin * mm_per_pixel_y, ymax * mm_per_pixel_y)

        cumulative_depths = np.cumsum(np.concatenate([[0], slice_depths]))
        z_min = cumulative_depths[zmin]
        z_max = cumulative_depths[min(zmax + 1, len(cumulative_depths) - 1)]
        bbox_z = (z_min, z_max)

        bbox_dimensions = (bbox_x[1] - bbox_x[0], bbox_y[1] - bbox_y[0], bbox_z[1] - bbox_z[0])

        return {'x': bbox_x, 'y': bbox_y, 'z': bbox_z, 'dimensions': bbox_dimensions}

    def calculate_density(self, volume: float, x_length_mm: float,
                          y_length_mm: float, total_depth_mm: float) -> float:
        """Calculate object density as percentage of total space (volume_calculator.py:96-100)."""
        total_possible_volume = x_length_mm * y_length_mm * total_depth_mm
        return volume / total_possible_volume

    def analyze_object_properties(self, voxel_data: np.ndarray, processed_volume: float,
                                  mesh_volume: float, surface_area: float,
                                  mm_per_pixel_x: float, mm_per_pixel_y: float,
                                  slice_depths: np.ndarray, x_length_mm: float,
                                  y_length_mm: float, total_depth_mm: float) -> dict:
        """Analyze comprehensive object properties with variable slice depths (volume_calculator.py:102-131)."""
        voxel_volume = self.calculate_voxel_volume_variable_depth(voxel_data, mm_per_pixel_x, mm_per_pixel_y, slice_depths)
        bbox_info = self.calculate_bounding_box_variable_depth(voxel_data, mm_per_pixel_x, mm_per_pixel_y, slice_depths)

        primary_volume = mesh_volume if mesh_volume is not None else processed_volume

        total_actual_depth = np.sum(slice_depths)
        density = self.calculate_density(primary_volume, x_length_mm, y_length_mm, total_actual_depth)

        print(f"Volume: {primary_volume:.4f} mm³")
        print(f"Dimensions: {bbox_info['dimensions'][0]:.2f} x {bbox_info['dimensions'][1]:.2f} x {bbox_info['dimensions'][2]:.2f} mm")
        if surface_area:
            print(f"Surface Area: {surface_area:.4f} mm²")
        print(f"Density: {100*density:.1f}% of total space")

        return {
            'volume_mm3': primary_volume,
            'voxel_volume_mm3': voxel_volume,
            'processed_voxel_volume_mm3': processed_volume,
            'mesh_volume_mm3': mesh_volume,
            'bounding_box': {'x': bbox_info['x'], 'y': bbox_info['y'], 'z': bbox_info['z']},
            'dimensions': bbox_info['dimensions'],
            'surface_area_mm2': surface_area,
            'density': density
        }

    # ------------------------------------------------------------------------------------------------
    # additive API (no reference counterpart)
    def analyze_components(self, voxel_data: np.ndarray, mm_per_pixel_x: float, mm_per_pixel_y: float,
                           slice_depths: np.ndarray, connectivity: int = 6) -> dict:
        """Per connected component (scipy.ndimage.label numbering, 6- or 26-connected), as arrays over the K components:
          n_components   K
          voxel_counts   int64 (K,)
          volume_mm3     float64 (K,): calculate_voxel_volume_variable_depth(labels == c, ...) bit for bit.  The float64 sums
                         run per component, so they need not add up bit-exactly to the volume of the whole grid.
          bbox_index     int32 (K, 6) [zmin, zmax, ymin, ymax, xmin, xmax], inclusive
          bbox_mm        float64 (K, 6) [z0, z1, y0, y1, x0, x1] and
          dimensions_mm  float64 (K, 3) [x, y, z] (the order of the reference's 'dimensions'): the values of
                         calculate_bounding_box_variable_depth(labels == c, ...), bit for bit; all zero when slice_depths is
                         empty.  Where that function would raise IndexError (a component whose first slice lies beyond
                         index len(slice_depths)), the z bounds and the z dimension are NaN.
        Prints nothing."""
        comps = engine.label_components(self._dv(voxel_data), connectivity)
        K = comps.n
        b = comps.bbox_index()
        bbox_mm = np.zeros((K, 6), dtype=np.float64)
        dims = np.zeros((K, 3), dtype=np.float64)
        if K and len(slice_depths):
            bi = b.astype(np.int64)
            bbox_mm[:, 4], bbox_mm[:, 5] = bi[:, 4] * mm_per_pixel_x, bi[:, 5] * mm_per_pixel_x
            bbox_mm[:, 2], bbox_mm[:, 3] = bi[:, 2] * mm_per_pixel_y, bi[:, 3] * mm_per_pixel_y
            cum = np.cumsum(np.concatenate([[0], slice_depths]))
            ok = bi[:, 0] < len(cum)
            bbox_mm[:, 0] = np.where(ok, cum[np.minimum(bi[:, 0], len(cum) - 1)], np.nan)
            bbox_mm[:, 1] = np.where(ok, cum[np.minimum(bi[:, 1] + 1, len(cum) - 1)], np.nan)
            dims[:, 0] = bbox_mm[:, 5] - bbox_mm[:, 4]
            dims[:, 1] = bbox_mm[:, 3] - bbox_mm[:, 2]
            dims[:, 2] = bbox_mm[:, 1] - bbox_mm[:, 0]
        return {
            'n_components': K,
            'voxel_counts': comps.counts(),
            'volume_mm3': comps.volumes_mm3(mm_per_pixel_x, mm_per_pixel_y, slice_depths),
            'bbox_index': b,
            'bbox_mm': bbox_mm,
            'dimensions_mm': dims,
        }
