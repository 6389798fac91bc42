"""Destroying a scene or a group gives back every device allocation the scene made, the lazily allocated ones included.

Each kind of scene is driven through every call that allocates on first use or grows a buffer: host traces below and above the
pipelined size (batch staging, pinned pipeline, cost and instance-id slots), hit attributes, three frames in flight with kept
rays and ray costs, the downloads (untile staging), both readback slots, geometry offsets, the refit topology and a TLAS
rebuild or set_instances that grows the node array."""
import numpy as np
import pytest

from conftest import random_rays
from test_build_reference import soup
from test_instances import xforms
from tray_racing_b200 import cuda, host

gpu = pytest.mark.gpu

N_OBJ, PER_OBJ = 250, 800                       # 200k triangles
W, H = 1024, 576                                # 589824 frame items: every per-item frame buffer spans at least 2 MiB
BIG = (1 << 19) + 4096                          # above the 2^18 rays of the pipelined host path; 2 MiB of instance ids
CAMERA = host.Camera((1.5, 1.1, 1.9), (0.0, 0.0, 0.0), 50.0)
FLAGS = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_KEEP_RAYS | cuda.RENDER_COUNTERS
PAGE = 2 << 20


def exercise(sc, instanced=False):
    """every lazily allocated buffer of a scene, the refits excepted"""
    for rays in (random_rays(5000, seed=1), random_rays(BIG, seed=2)):
        hits, ids = sc.traverse_instance(rays) if instanced else (sc.traverse(rays), None)
        sc.traverse_cost(rays)
        sc.hit_attributes(rays, hits, ids)
    sc.set_frames_in_flight(3)
    sc.set_ray_cost(True)
    view = host.view_from_camera(CAMERA, W, H, sc.info()["tlas_start"])
    for fc in range(3):
        sc.render(view, W, H, fc, FLAGS)
    sc.sync()
    sc.download(primary=True, bounce=True, bounce_rays=True, rgba=True)
    sc.download_cost(primary=True, bounce=True)
    sc.download_attributes(primary=True, bounce=True)
    if instanced:
        sc.download_instance(primary=True, bounce=True)
    rgba = [np.zeros((H, W, 4), np.uint8) for _ in range(2)]
    for slot in (0, 1):
        sc.readback_begin(rgba[slot], slot)
    for slot in (0, 1):
        sc.readback_wait(slot)
    sc.set_geometry_offsets(np.arange(N_OBJ + 1, dtype=np.uint32) * PER_OBJ)
    sc.hits_to_geometry(hits)


def cycle(tris, offsets):
    """create, exercise and destroy a created flat scene, a device-built two-level scene, the same created from its bytes, the
    built one instanced, and a one-device group"""
    moved = np.ascontiguousarray(tris * np.float32(1.01))
    src = cuda.TrayCudaScene.build(tris)
    nodes, rec, prim = src.download_bvh()
    src.close()
    flat = cuda.TrayCudaScene(nodes, rec, 48)
    try:
        exercise(flat)
        flat.refit(moved[prim])
    finally:
        flat.close()

    built = cuda.TrayCudaScene.build(tris, object_offsets=offsets)
    try:
        exercise(built)
        built.refit(moved)
        built.refit_rebuild_tlas(moved)
        nodes2, rec2, prim2 = built.download_bvh()
        blas, ts = built.download_instances(), built.info()["tlas_start"]
    finally:
        built.close()
    created = cuda.TrayCudaScene(nodes2, rec2, 48, blas, ts)      # holds n_nodes: the TLAS rebuild grows its node array
    try:
        exercise(created)
        created.refit_rebuild_tlas(moved[prim2])
    finally:
        created.close()

    inst = cuda.TrayCudaScene.build(tris, object_offsets=offsets)
    try:
        roots = np.unique(inst.download_instances())
        n = 2 * N_OBJ                                               # more instances than objects: the node array grows
        inst.set_instances(np.random.default_rng(3).choice(roots, n), xforms("mixed", n, 3))
        exercise(inst, instanced=True)
        inst.refit_rebuild_tlas(moved)
    finally:
        inst.close()

    grp = cuda.TrayCudaGroup(nodes, rec, 48, devices=[0])
    try:
        grp.set_frames_in_flight(2)
        for fc in range(3):
            grp.render(host.view_from_camera(CAMERA, W, H), W, H, fc)
        grp.frame()
    finally:
        grp.close()


@gpu
def test_destroy_gives_back_every_allocation():
    """Four cycles of `cycle`: the first loads the kernels and lets the driver set up what it keeps for the context; after each
    of the other three, once the device is synchronised, free device memory is not below what it was after the first by more
    than one 2 MiB page.  Device memory is mapped in 2 MiB pages and the driver sub-allocates small requests from pages it
    keeps, so a leak of a few words need not show; every buffer sized by the triangles, the rays or the frame spans more than a
    page here, so a leak of any of them takes more than the slack in one cycle.  Only device memory is measured: pinned host
    memory, streams and events are not covered."""
    import torch
    tris = soup(N_OBJ * PER_OBJ, seed=29)
    offsets = np.arange(N_OBJ + 1, dtype=np.uint64) * PER_OBJ
    cycle(tris, offsets)
    torch.cuda.synchronize()
    free = torch.cuda.mem_get_info()[0]
    lost = []
    for _ in range(3):
        cycle(tris, offsets)
        torch.cuda.synchronize()
        lost.append(free - torch.cuda.mem_get_info()[0])
    assert max(lost) <= PAGE, f"device bytes not given back after each cycle: {lost}"
