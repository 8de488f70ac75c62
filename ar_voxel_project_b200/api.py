"""The reference's free functions for the hot path, same names and argument meaning:

    carve / fastCarve                     VoxelCarving.h:19,31
    reconstructClosestColor / AvgColor    ColorReconstruction.h:131,142
    marchingCubesClassify                 the cube-index half of marchingCubes, MarchingCubes.h:596

The reference passes (cameraMatrix, distCoeffs, model, images, masks) and re-estimates poses and
re-undistorts inside every call (VoxelCarving.cpp:25,36; ColorReconstruction.h:17-28).  Here those
host-side, once-per-dataset results arrive cached in a ViewSet; everything else (Model in, Model
mutated in place, nothing retained) is unchanged.  Errors raise VoxCarveError where the reference
prints to std::cerr and returns.
"""
import numpy as np

from . import _lib as L
from .engine import VoxelEngine
from .model import Model


class ViewSet:
    """Cached per-dataset inputs (SURVEY §7-1): P = K32*pose, M = pose (3x4 world->camera),
    undistorted silhouettes (bit-packed, 1 = background) and undistorted BGR images."""

    def __init__(self, P, M, W, H, mask_bits=None, mask_bgr=None, images_bgr=None):
        self.P = np.ascontiguousarray(P, np.float32).reshape(-1, 3, 4)
        self.M = None if M is None else np.ascontiguousarray(M, np.float32).reshape(-1, 3, 4)
        self.W, self.H = int(W), int(H)
        self.mask_bits, self.mask_bgr, self.images_bgr = mask_bits, mask_bgr, images_bgr
        if mask_bits is None and mask_bgr is None:
            raise ValueError("ViewSet needs masks")
        n_masks = len(mask_bits) if mask_bits is not None else len(mask_bgr)
        if n_masks != len(self.P):
            raise ValueError("Number of images doesn't match number of masks.")  # main.cpp:228-231

    @property
    def V(self):
        return len(self.P)

    @classmethod
    def from_npz(cls, path, with_images=True):
        """tests/golden/*_views.npz written by tools/make_goldens.py"""
        z = np.load(path)
        imgs = None
        if with_images:
            import cv2  # PNG decode only
            off = z["png_offsets"]
            imgs = np.stack([cv2.imdecode(z["png_blob"][off[i]:off[i + 1]], 1) for i in range(int(z["V"]))])
        return cls(z["P"], z["M"], int(z["W"]), int(z["H"]), mask_bits=z["mask_bits"], images_bgr=imgs)


def _engine_for(model, views, device=0, need_images=False):
    """an engine holding all views: vc_set_views takes the first 256, vc_append_views the rest"""
    if need_images and views.images_bgr is None:
        raise ValueError("colour reconstruction needs the undistorted images")
    e = VoxelEngine(model.getX(), model.getY(), model.getZ(), model.getSize(), device=device)
    k = min(views.V, 256)
    e.set_views(views.P[:k], views.W, views.H, None if views.M is None else views.M[:k])
    if views.mask_bits is not None:
        e.set_masks_bits(views.mask_bits[:k])
    else:
        e.set_masks_bgr(views.mask_bgr[:k])
    if need_images:
        e.set_images(views.images_bgr[:k])
    if views.V > k:
        e.append_views(views.P[k:], None if views.M is None else views.M[k:],
                       mask_bits=None if views.mask_bits is None else views.mask_bits[k:],
                       mask_bgr=None if views.mask_bits is not None else views.mask_bgr[k:],
                       images_bgr=views.images_bgr[k:] if need_images else None)
    return e


def carve(views, model, intermediateMeshes=False, mode=L.VC_EXACT, device=0):
    """carve() VoxelCarving.cpp:60-72. Returns per-view (hist, n_active, n_tris) if intermediateMeshes."""
    print("LOG - VC: starting carving process (version 1).")
    inter = []
    with _engine_for(model, views, device) as e:
        if intermediateMeshes:  # :65-68 — a cube-index pass after every view
            for v in range(views.V):
                e.carve(mode, v, v + 1)
                e.mc_classify()
                inter.append(e.download_mc())
        else:
            e.carve(mode)
        model.apply_carve(e.download_occupied(), e.download_seen())
    print("LOG - VC: carving complete.")
    return inter if intermediateMeshes else None


def fastCarve(views, model, mode=L.VC_EXACT, device=0):
    """fastCarve() VoxelCarving.cpp:74-167."""
    print("LOG - VC: starting carving process (version 2).")
    with _engine_for(model, views, device) as e:
        e.fast_carve(mode)
        model.apply_carve(e.download_occupied(), e.download_seen())
    print("LOG - VC: carving complete.")


def _upload_model(e, model):
    """occupancy of an already-carved host Model -> engine volumes (colour / MC read the device grid)."""
    from .synth import pack_bits
    import ctypes as C
    occ = pack_bits(model.occupied_grid())
    seen = pack_bits(model.seen.reshape(model.getZ(), model.getY(), model.getX()))
    e.upload_volumes(occ, seen)


def _color(views, model, mode, device):
    with _engine_for(model, views, device, need_images=True) as e:
        _upload_model(e, model)
        e.color(mode)
        idx, rgbn = e.download_colors()
    model.apply_colors(idx, rgbn)


def reconstructClosestColor(views, model, device=0):
    """ColorReconstruction.cpp:22-46"""
    print("LOG - CR: starting color reconstruction (closest color).")
    _color(views, model, L.VC_COLOR_CLOSEST, device)
    print("LOG - CR: color reconstruction finished.")


def reconstructAvgColor(views, model, device=0):
    """ColorReconstruction.cpp:48-70"""
    print("LOG - CR: starting color reconstruction (average color).")
    _color(views, model, L.VC_COLOR_AVG, device)
    print("LOG - CR: color reconstruction finished.")


def marchingCubesClassify(model, device=0):
    """cube-index classification of marchingCubes() (MarchingCubes.cpp:12-18, MarchingCubes.h:479-488):
    -> (hist[256], n_active_cells, n_triangles)"""
    print("LOG - MC: starting to process Voxels.")
    with VoxelEngine(model.getX(), model.getY(), model.getZ(), model.getSize(), device=device) as e:
        _upload_model(e, model)
        e.mc_classify()
        out = e.download_mc()
    print("LOG - MC: voxel processing completed.")
    return out
