"""CPU checks of the connected-components reference that tests/test_gpu_components.py compares the GPU against:
scipy's labels canonicalised to the id rule of include/scan3d.h (rank of the smallest vertex) agree with a plain
union-find, and the keep rule and the compaction follow the header.  The new C entries reject null arguments without
a GPU."""
import ctypes as C

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from gpu_common import s3


def labels_ref(faces, n):
    """(int32 labels [n], component count): scipy's components, ids ranked by their smallest vertex"""
    faces = np.asarray(faces, np.int64).reshape(-1, 3)
    if n == 0:
        return np.zeros(0, np.int32), 0
    rows = np.concatenate([faces[:, 0], faces[:, 0]])
    cols = np.concatenate([faces[:, 1], faces[:, 2]])
    g = coo_matrix((np.ones(len(rows), np.int8), (rows, cols)), shape=(n, n))
    c, lab = connected_components(g, directed=False)
    first = np.full(c, n, np.int64)
    np.minimum.at(first, lab, np.arange(n))
    rank = np.empty(c, np.int64)
    rank[np.argsort(first)] = np.arange(c)
    return rank[lab].astype(np.int32), c


def keep_ref(labels, faces, c, min_faces, max_components):
    """(vertices [c], faces [c], kept bool [c]) of the keep rule"""
    fl = labels[faces[:, 0]] if len(faces) else np.zeros(0, np.int64)
    vcount = np.bincount(labels, minlength=c).astype(np.int64)
    fcount = np.bincount(fl, minlength=c).astype(np.int64)
    ids = np.flatnonzero(fcount >= min_faces)
    ids = ids[np.lexsort((ids, -fcount[ids]))]          # faces descending, then the smaller id
    if max_components:
        ids = ids[:max_components]
    kept = np.zeros(c, bool)
    kept[ids] = True
    return vcount, fcount, kept


def compact_ref(mesh, labels, kept):
    """the header's compaction: new = cumsum(keep_v) - 1; faces = new[faces[keep_f]]"""
    xyz, nrm, rgb, faces = mesh
    keep_v = kept[labels]
    keep_f = kept[labels[faces[:, 0]]] if len(faces) else np.zeros(0, bool)
    new = np.cumsum(keep_v) - 1
    return xyz[keep_v], nrm[keep_v], rgb[keep_v], new[faces[keep_f]].astype(np.int32).reshape(-1, 3)


def random_mesh(rng, n, groups, faces_per_group, isolated=0):
    """a mesh of `groups` pieces over a random permutation of n vertices, `isolated` of them in no face, with
    duplicate and degenerate faces"""
    perm = rng.permutation(n)
    used, free = perm[:n - isolated], perm[n - isolated:]
    parts = np.array_split(used, groups)
    out = []
    for p in parts:
        if len(p) == 0:
            continue
        chain = np.stack([p, np.roll(p, -1), np.roll(p, -2)], 1)     # every vertex of the piece in some face
        extra = p[rng.integers(0, len(p), (faces_per_group, 3))]
        out += [chain, extra]
        a = p[rng.integers(0, len(p))]
        b = p[rng.integers(0, len(p))]
        out += [np.array([[a, a, b], [a, a, a]]), extra[:3]]        # degenerate and duplicate faces
    faces = np.concatenate(out).astype(np.int32)
    return faces[rng.permutation(len(faces))], free


def _union_find(faces, n):
    parent = list(range(n))

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a
    for a, b, c in faces:
        for x in (b, c):
            ra, rx = find(a), find(x)
            if ra != rx:
                parent[max(ra, rx)] = min(ra, rx)
    roots = sorted({find(v) for v in range(n)})
    rank = {r: i for i, r in enumerate(roots)}
    return np.array([rank[find(v)] for v in range(n)], np.int32), len(roots)


@pytest.mark.parametrize("seed", range(4))
def test_reference_labels_follow_the_id_rule(seed):
    rng = np.random.default_rng(seed)
    faces, free = random_mesh(rng, 3000, 1 + seed * 7, 40, isolated=25)
    lab, c = labels_ref(faces, 3000)
    want, cw = _union_find(faces, 3000)
    assert c == cw and np.array_equal(lab, want)
    assert lab[0] == 0 and (lab[free] >= 0).all()
    first = np.array([np.flatnonzero(lab == k)[0] for k in range(c)])
    assert (np.diff(first) > 0).all()                   # ids ranked by the smallest vertex


def test_reference_keep_rule_and_compaction():
    # components {0, 1, 2} (2 faces), {3} (no face), {4, 5, 6} (3 faces), {7, 8, 9} (2 faces)
    faces = np.array([[0, 1, 2], [2, 1, 0], [4, 5, 6], [6, 6, 4], [5, 4, 4], [7, 8, 9], [9, 8, 7]], np.int32)
    lab, c = labels_ref(faces, 10)
    assert c == 4 and list(lab) == [0, 0, 0, 1, 2, 2, 2, 3, 3, 3]
    assert keep_ref(lab, faces, c, 0, 0)[2].tolist() == [True, True, True, True]
    assert keep_ref(lab, faces, c, 1, 0)[2].tolist() == [True, False, True, True]
    assert keep_ref(lab, faces, c, 3, 0)[2].tolist() == [False, False, True, False]
    assert keep_ref(lab, faces, c, 0, 2)[2].tolist() == [True, False, True, False]    # the tie goes to id 0
    v, f, kept = keep_ref(lab, faces, c, 0, 1)
    assert v.tolist() == [3, 1, 3, 3] and f.tolist() == [2, 0, 3, 2] and kept.tolist() == [False, False, True, False]
    xyz = np.arange(30, dtype=np.float32).reshape(10, 3)
    mesh = (xyz, -xyz, xyz.astype(np.uint8), faces)
    out = compact_ref(mesh, lab, kept)
    assert np.array_equal(out[0], xyz[4:7]) and out[3].tolist() == [[0, 1, 2], [2, 2, 0], [1, 0, 0]]


def test_component_entries_reject_null_arguments_without_a_gpu():
    L = s3.cuda_lib()
    p, r, n = s3.ComponentsParams(0, 0), s3.ComponentsResultC(), C.c_int64()
    assert L.scan3d_voxel_surface_components(None, C.byref(p), C.byref(r)) == -4
    assert L.scan3d_get_surface_components(None, None, None, None, 0) == -4
    assert L.scan3d_mesh_components_dev(None, None, 0, 0, None, C.byref(n)) == -4
