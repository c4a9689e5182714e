"""Drop-in for the numerical part of the reference's 3D_clustering/region_growing.py (`rg`;
SURVEY.md section 8f, N4): same function names, arguments, prints and return types.

    get_vertex_info / get_pos / generate_sphere_ply / set_clusters / set_normal    rg:11-76, :224-261 (PLY helpers)
    compute_normals(V1, k)                   rg:78-127   -> float64 [N, 3]
    compute_residuals(V1, normals, k)        rg:130-163  -> float64 [N]
    segmentation_3D(points, normals, residuals, residual_threshold, angle_threshold, k)   rg:166-221
                                             -> list of regions (lists of point indices), largest first

Neighbour search, centroids, covariance, eigenvectors and residuals run on the GPU through
libgslift.so (gsl_region_knn_pca, csrc/region_growing.cu); the growth loop is serial by
construction and runs on the host inside the library (gsl_region_grow) over neighbour lists the
GPU produced.  There is no CPU path for the numerical part.
"""
from __future__ import annotations

import math
import random

import numpy as np
import torch

from . import ops, plyio
from ._native import check, lib


def _device_points(V1) -> torch.Tensor:
    if isinstance(V1, torch.Tensor):
        t = V1.to(torch.float32)
    else:
        t = torch.from_numpy(np.ascontiguousarray(V1, np.float32))
    if t.dim() != 2 or t.shape[1] != 3:
        raise ValueError("points must have shape (N, 3)")
    if not torch.cuda.is_available():
        raise RuntimeError("region_growing needs a CUDA device (there is no CPU path)")
    t = t.cuda().contiguous()
    if not bool(torch.isfinite(t).all()):
        raise ValueError("data must be finite, check for nan or inf values")      # scipy KDTree's message
    return t


def knn_pca(V1, k: int, normals_in=None, want_normals=True, want_residuals=True, want_centroids=False,
            want_knn=False, want_stats=False) -> dict:
    """One pass of gsl_region_knn_pca.  Returns device tensors: normals f64 [N,3], residuals f64 [N],
    centroids f64 [N,3], knn int32 [N,k] in increasing (distance, index) order, as requested.  Lists are
    returned for k <= GSL_REGION_MAX_LIST (16384); above that want_knn raises the library's GslError."""
    pos = _device_points(V1)
    N = pos.shape[0]
    dev = pos.device
    out = {}
    nin = None
    if normals_in is not None:
        nin = (normals_in if isinstance(normals_in, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(normals_in, np.float64)))
        nin = nin.to(dev, torch.float64).contiguous()
        if tuple(nin.shape) != (N, 3):
            raise ValueError("normals must have shape (N, 3)")
    if want_normals:
        out["normals"] = torch.empty((N, 3), dtype=torch.float64, device=dev)
    if want_residuals:
        out["residuals"] = torch.empty(N, dtype=torch.float64, device=dev)
    if want_centroids:
        out["centroids"] = torch.empty((N, 3), dtype=torch.float64, device=dev)
    if want_knn:
        out["knn"] = torch.empty((N, int(k)), dtype=torch.int32, device=dev)
    if want_stats:          # [walks over candidate cells, points visited, cubes too small, further select walks]
        out["stats"] = torch.zeros(4, dtype=torch.int64, device=dev)
    L = lib()
    ws = ops._ws.get(dev, L.gsl_region_workspace_bytes(N))
    ptr = lambda name: out[name].data_ptr() if name in out else None
    with torch.cuda.device(dev):
        check(L.gsl_region_knn_pca(pos.data_ptr(), N, int(k), nin.data_ptr() if nin is not None else None, ptr("normals"),
                                   ptr("residuals"), ptr("centroids"), ptr("knn"), ptr("stats"), ws.data_ptr(), ws.numel(), ops._stream()))
    return out


def compute_normals(V1, k):
    """Compute normals using PCA on k-nearest neighbors (rg:78-127).  Returns float64 (N, 3)."""
    print("Calculating normals...")
    n = len(V1)
    for i in range(0, n, 1000):                     # the reference's progress lines (rg:96-97)
        print(f"Processing point {i}/{n}")
    normals = knn_pca(V1, k, want_residuals=False)["normals"].cpu().numpy()
    print("Normal calculation complete.")
    return normals


def compute_residuals(V1, normals, k):
    """Residuals: orthogonal distance of every point to the plane through its neighbours' centroid
    (rg:130-163).  Returns float64 (N,)."""
    print("Calculating residuals...")
    n = len(V1)
    for i in range(0, n, 1000):                     # rg:149-150
        print(f"Processing point {i}/{n}")
    return knn_pca(V1, k, normals_in=normals, want_normals=False)["residuals"].cpu().numpy()


def segmentation_3D(points, normals, residuals, residual_threshold, angle_threshold, k):
    """Region growing with the smoothness constraint (rg:166-221).  Returns the list of regions
    (each a list of point indices), sorted by size, largest first (rg:219)."""
    knn = knn_pca(points, k, want_normals=False, want_residuals=False, want_knn=True)["knn"].cpu().numpy()
    normals = np.ascontiguousarray(normals, np.float64)
    residuals = np.ascontiguousarray(residuals, np.float64)
    n = knn.shape[0]
    region_of = np.empty(n, np.int32)
    sizes = np.empty(max(n, 1), np.int64)
    r = lib().gsl_region_grow(knn.ctypes.data, int(k), normals.ctypes.data, residuals.ctypes.data, n,
                              float(residual_threshold), float(angle_threshold), region_of.ctypes.data, sizes.ctypes.data)
    if r < 0:
        check(int(r))
    order = np.argsort(region_of, kind="stable")
    bounds = np.concatenate(([0], np.cumsum(sizes[:r])))
    regions = [order[bounds[i]:bounds[i + 1]].tolist() for i in range(int(r))]
    regions.sort(key=len, reverse=True)             # rg:219 (stable, like list.sort)
    return regions


# --------------------------------------------------------------------------------------
# PLY helpers of the script (host side; plyfile is replaced by plyio)
# --------------------------------------------------------------------------------------
def get_vertex_info(plydata):
    """(points [N,3], colors [N,3]) = (x, y, z), (f_dc_0..2) of the vertex element (rg:11-30)."""
    vertices = plydata["vertex"]
    points = np.column_stack((vertices["x"], vertices["y"], vertices["z"]))
    colors = np.column_stack((vertices["f_dc_0"], vertices["f_dc_1"], vertices["f_dc_2"]))
    return points, colors


def get_pos(plydata):
    """Positions [N,3] of the vertex element (rg:32-40; the reference reads the global `plydata`)."""
    vertices = plydata["vertex"]
    return np.column_stack((vertices["x"], vertices["y"], vertices["z"]))


def generate_sphere_ply(radius=1.0, subdivisions=50, filename="sphere.ply"):
    """ASCII PLY of a red latitude / longitude sphere (rg:42-76), same text byte for byte."""
    vertices = []
    for i in range(subdivisions + 1):
        theta = i * math.pi / subdivisions
        for j in range(subdivisions):
            phi = j * 2.0 * math.pi / subdivisions
            vertices.append([radius * math.sin(theta) * math.cos(phi), radius * math.sin(theta) * math.sin(phi),
                             radius * math.cos(theta), 255, 0, 0])
    vertices = np.array(vertices)
    with open(filename, "w") as ply_file:
        ply_file.write("ply\nformat ascii 1.0\n")
        ply_file.write(f"element vertex {len(vertices)}\n")
        ply_file.write("property float x\nproperty float y\nproperty float z\n")
        ply_file.write("property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")
        for v in vertices:
            ply_file.write(f"{v[0]:.6f} {v[1]:.6f} {v[2]:.6f} {int(v[3])} {int(v[4])} {int(v[5])}\n")
    print(f"Sphere saved to {filename}")


def set_clusters(plydata, R, modified_path):
    """One random colour per region into f_dc_0..2, then write the PLY in the input's format (rg:224-241)."""
    vertices = plydata["vertex"]
    for Rc in R:
        r = np.array(Rc)
        vertices["f_dc_0"][r] = random.random()
        vertices["f_dc_1"][r] = random.random()
        vertices["f_dc_2"][r] = random.random()
    with open(modified_path, "wb") as f:
        print("writing new data")
        plydata.write(f)


def set_normal(plydata, normals, modified_path):
    """Normals into the diffuse colour channels, then write the PLY (rg:244-261)."""
    vertices = plydata["vertex"]
    vertices["f_dc_0"] = normals[:, 0]
    vertices["f_dc_1"] = normals[:, 1]
    vertices["f_dc_2"] = normals[:, 2]
    print(normals[:, 0] * 255)
    with open(modified_path, "wb") as f:
        print("writing new data")
        plydata.write(f)


def main(file_path=r"data\point_cloud.ply", modified_path=r"3D_clustering\clustering.ply"):
    """The script's __main__ (rg:263-285) with its constants: k = 2000 for normals and residuals,
    residual_threshold 0.1, angle_threshold 0.05, k = 10 for the growth."""
    with open(file_path, "rb") as f:
        plydata = plyio.read_ply(f)
    points = get_pos(plydata)
    normals = compute_normals(points, 2000)
    residuals = compute_residuals(points, normals, 2000)
    print(residuals)
    R = segmentation_3D(points, normals, residuals, residual_threshold=0.1, angle_threshold=0.05, k=10)
    print(f"number of segments: {len(R)}")
    set_clusters(plydata, R, modified_path)
    return R


if __name__ == "__main__":
    import sys
    main(*sys.argv[1:3])
