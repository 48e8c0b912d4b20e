"""``MembraneMesh`` facade: the reference's block driver and curvature properties on top of the GPU
solver (reference: ``ch_shrinkwrap/_membrane_mesh.pyx``).

The drop-in boundary sits at ``_membrane_mesh.pyx:1510-1517`` (one ``ShrinkwrapMeshConjGrad`` per remesh
block) and at ``curvature_grad_c`` (``:323-347``).  Everything topological -- remesh, neck removal, hole
punching, repair -- stays on the host in the mesh class's own methods (PYME's ``TriangleMesh`` in the
reference, SURVEY section 0.2); this module only calls them when the host mesh provides them.

``ShrinkwrapMeshMixin`` can be mixed into any half-edge mesh exposing PYME's structured arrays
(``_vertices``, ``_faces``, ``_halfedges``, ``faces``, ``vertex_normals`` ...); ``MembraneMesh`` below
combines it with the harness mini-mesh so tests and bench.py can run the whole driver without PYME.
"""
from __future__ import annotations

import ctypes
import logging
import math

import numpy as np

from . import _lib
from .mesh_conj_grad import ShrinkwrapMeshConjGrad, _session_for
from .minimesh import MiniMesh

logger = logging.getLogger(__name__)

KBT = 0.0257   # membrane_mesh_utils.h:16

DESCENT_METHODS = ['conjugate_gradient']
DEFAULT_DESCENT_METHOD = 'conjugate_gradient'

_CURV_SCALARS = ('k0', 'k1', 'H', 'K', 'dH', 'dK', 'E', 'pE', 'dE_neighbors')
_CURV_VECTORS = ('e0', 'e1', 'dEdN')


def curvature_grad(mesh, dN=0.1, skip_prob=0.0, kc=1.0, kg=-20.0 * KBT, c0=0.0, jitter_u=None, seed=0,
                   out=None, device=0):
    """``c_curvature_grad`` (membrane_mesh_utils.c:915-1250) on the GPU through nw_curvature_grad.

    Returns a dict of float32 arrays: k0,k1,H,K,dH,dK,E,pE,dE_neighbors (M,) and e0,e1,dEdN (M,3).
    ``out`` may supply preallocated arrays (the reference overwrites caller-owned buffers in place).
    """
    sess = _session_for(mesh, device)
    M = len(mesh._vertices)
    res = out if out is not None else {}
    for k in _CURV_SCALARS:
        if k not in res:
            res[k] = np.zeros(M, np.float32)
    for k in _CURV_VECTORS:
        if k not in res:
            res[k] = np.zeros((M, 3), np.float32)
    verts = np.ascontiguousarray(mesh._vertices)
    faces = np.ascontiguousarray(mesh._faces)
    hes = np.ascontiguousarray(mesh._halfedges)
    if verts.dtype.itemsize != 120 or faces.dtype.itemsize != 24 or hes.dtype.itemsize != 28:
        raise RuntimeError('mesh record layouts differ from membrane_mesh_utils.h:31-65')
    ju = None if jitter_u is None else np.ascontiguousarray(jitter_u, dtype=np.float64)
    if ju is not None and ju.size < 3 * int((verts['halfedge'] != -1).sum()):
        raise ValueError('jitter_u needs 3 values per valid vertex')
    f = _lib.fptr
    sess.handle.call('nw_curvature_grad', ctypes.c_void_p(verts.ctypes.data), ctypes.c_void_p(faces.ctypes.data),
                     ctypes.c_void_p(hes.ctypes.data), int(M), int(len(faces)), int(len(hes)), float(dN), float(skip_prob),
                     f(res['k0']), f(res['k1']), f(res['e0']), f(res['e1']), f(res['H']), f(res['K']), f(res['dH']), f(res['dK']),
                     f(res['E']), f(res['pE']), f(res['dE_neighbors']), float(kc), float(kg), float(c0), f(res['dEdN']),
                     _lib.dptr(ju), int(seed))
    return res


def neck_candidates(mesh, low, high, device=0):
    """``np.flatnonzero((K < low) | (K > high))`` on the K of the last curvature call (_membrane_mesh.pyx:1212-1213)."""
    sess = _session_for(mesh, device)
    n = ctypes.c_int(0)
    sess.handle.call('nw_neck_candidates', float(low), float(high), None, ctypes.byref(n))
    idx = np.empty(max(n.value, 1), np.int32)
    sess.handle.call('nw_neck_candidates', float(low), float(high), _lib.iptr(idx), ctypes.byref(n))
    return idx[:n.value]


class ShrinkwrapMeshMixin:
    """Parameters and methods of the reference ``MembraneMesh`` that lie on the NanoWrap path."""

    def _init_shrinkwrap(self, **kwargs):
        # _membrane_mesh.pyx:82-120
        self.kc = 20.0 * KBT
        self.kg = -20.0 * KBT
        self.c0 = 0.0
        self.step_size = 1
        self.beta_1, self.beta_2, self.eps = 0.8, 0.7, 1e-8
        self.max_iter = 250
        self.remesh_frequency = 100
        self.delaunay_remesh_frequency = 150
        self.delaunay_eps = 100.0
        self.search_k = 200
        self.search_rad = 100
        self.skip_prob = 0.0
        self.shrink_weight = 0
        self.smooth_curvature = False
        self.cg = None
        self._points = None
        self._sigma = None
        self._initialize_curvature_vectors()
        for key, value in kwargs.items():
            setattr(self, key, value)

    # -- curvature cache (_membrane_mesh.pyx:122-214) ---------------------------------------------------
    _CURV_ATTRS = ('_H', '_K', '_E', '_k_0', '_k_1', '_e_0', '_e_1', '_pE', '_dH', '_dK', '_dE_neighbors')

    def _initialize_curvature_vectors(self):
        """_membrane_mesh.pyx:122-160: the cached curvature arrays are zeroed.  The solver calls this after EVERY iteration
        (mesh_conj_grad.py:290); allocating eleven M-sized arrays each time costs 2.5 ms at M = 5e5, so the arrays are only
        dropped here and re-created (zeroed) when something reads or fills them."""
        for name in self._CURV_ATTRS:
            self.__dict__.pop(name, None)

    def __getattr__(self, name):
        # only reached when the attribute is missing: the lazily re-created curvature caches
        if name in ShrinkwrapMeshMixin._CURV_ATTRS:
            sz = self._vertices.shape[0]
            arr = np.zeros((sz, 3) if name in ('_e_0', '_e_1') else sz, np.float32)
            self.__dict__[name] = arr
            return arr
        raise AttributeError(name)

    def curvature_grad_c(self, dN=0.1, skip_prob=0.0):
        """_membrane_mesh.pyx:323-347: fills the cached curvature arrays in place, returns dEdN."""
        out = dict(k0=self._k_0, k1=self._k_1, e0=self._e_0, e1=self._e_1, H=self._H, K=self._K, dH=self._dH, dK=self._dK,
                   E=self._E, pE=self._pE, dE_neighbors=self._dE_neighbors)
        res = curvature_grad(self, dN=dN, skip_prob=skip_prob, kc=self.kc, kg=self.kg, c0=self.c0, out=out,
                             seed=getattr(self, '_jitter_seed', 0))
        return res['dEdN']

    def _populate_curvature_grad(self):
        self.curvature_grad_c()
        if not getattr(self, 'smooth_curvature', False):
            return
        if hasattr(self, 'smooth_per_vertex_data'):      # PYME-side smoothing (:182-186), host code of the mesh class
            self._H = self.smooth_per_vertex_data(self._H)
            self._K = self.smooth_per_vertex_data(self._K)
            self._k_0 = self.smooth_per_vertex_data(self._k_0)
            self._k_1 = self.smooth_per_vertex_data(self._k_1)
            self._curvature_smoothing = 'host smooth_per_vertex_data'
        else:
            # PYME's TriangleMesh.smooth_per_vertex_data is not part of the reference repository (SURVEY 8c: unpinned);
            # without it the curvatures stay unsmoothed -- say so instead of skipping silently
            self._curvature_smoothing = 'skipped: the host mesh class has no smooth_per_vertex_data'
            logger.warning('smooth_curvature=True but %s has no smooth_per_vertex_data (PYME TriangleMesh method): '
                           'curvatures are left unsmoothed', type(self).__name__)

    def _lazy(self, name):
        if not np.any(getattr(self, name)):
            self._populate_curvature_grad()
        return getattr(self, name)

    @property
    def E(self):
        e = self._lazy('_E'); e[np.isnan(e)] = 0; return e

    @property
    def pE(self):
        e = self._lazy('_pE'); e[np.isnan(e)] = 0; return e

    curvature_principal0 = property(lambda self: self._lazy('_k_0'))
    curvature_principal1 = property(lambda self: self._lazy('_k_1'))
    eigenvector_principal0 = property(lambda self: self._lazy('_e_0'))
    eigenvector_principal1 = property(lambda self: self._lazy('_e_1'))
    curvature_mean = property(lambda self: self._lazy('_H'))
    curvature_gaussian = property(lambda self: self._lazy('_K'))

    # -- optimiser diagnostics (_membrane_mesh.pyx:1563-1634) --------------------------------------------
    @property
    def _S0(self):
        return self.cg.Ahfunc(self.cg.res).reshape(self.vertices.shape)

    S0 = property(lambda self: self.cg.S[:, 0].reshape(self.vertices.shape))
    S1 = property(lambda self: self.cg.S[:, 1].reshape(self.vertices.shape))
    S2 = property(lambda self: self.cg.S[:, 2].reshape(self.vertices.shape))

    @property
    def point_dis(self):
        s0 = self._S0
        return np.sqrt((s0 * s0).sum(1))

    def point_surface_distance(self, points=None, return_face=False, return_closest=False, signed=False):
        """Exact distance from each localisation to the fitted surface (float64); ``points=None``: the fit's own localisations
        (resident on the device).  Unlike ``point_dis``, which is per vertex and built from the fit's residuals, this is per
        point and measures the closed triangles.  ``signed=True``: negative inside the fitted surface, positive outside.  See
        ``ShrinkwrapMeshConjGrad.surface_distance``."""
        if self.cg is None:
            raise RuntimeError('point_surface_distance: no fit on this mesh yet (self.cg is None)')
        return self.cg.surface_distance(points, return_face=return_face, return_closest=return_closest, signed=signed)

    def self_intersections(self, return_stats=False):
        """The pairs of faces of the fitted surface that cross or touch beyond their shared vertices and edges ((n, 2) int32
        rows of ``faces``); see ``evaluation_utils.self_intersections``.  Runs on the fit's handle, nothing is uploaded."""
        if self.cg is None:
            raise RuntimeError('self_intersections: no fit on this mesh yet (self.cg is None)')
        return self.cg.self_intersections(return_stats=return_stats)

    @property
    def rms_point_sc(self):
        res = self.cg.res
        rn = (np.sqrt((res * res).reshape(-1, 3).sum(1))[:, None] * np.ones(3)[None, :]).ravel()
        rme = self.cg.Ahfunc(rn).reshape(self.vertices.shape)
        return np.sqrt((rme * rme).sum(1))

    @property
    def point_influence(self):
        fn = getattr(self.cg, 'point_influence', None)
        if callable(fn):                  # GPU solver: one fused pass on the device
            return fn()
        # any other solver object (the reference's, the oracle's): _membrane_mesh.pyx:1625-1634 as written
        s = self.cg.Ahfunc(np.ones_like(self.cg.res)).reshape(self.vertices.shape)
        return np.sqrt((s * s).sum(1))

    # -- neck removal: criterion on the GPU, topology on the host (_membrane_mesh.pyx:1201-1219) -------------
    def remove_necks(self, neck_curvature_threshold_low=-1e-4, neck_curvature_threshold_high=1e-2):
        self._populate_curvature_grad()
        if self.smooth_curvature and hasattr(self, 'smooth_per_vertex_data'):
            verts = np.flatnonzero((self._K < neck_curvature_threshold_low) | (self._K > neck_curvature_threshold_high))
        else:
            verts = neck_candidates(self, neck_curvature_threshold_low, neck_curvature_threshold_high)
        self._last_neck_candidates = verts
        if len(verts) > 0 and hasattr(self, 'unsafe_remove_vertices'):
            self.unsafe_remove_vertices(verts)
            self.repair()
            self.remesh(n_relax=0)
            self.remove_inner_surfaces()
        return verts

    # -- hole punching: the two searches on the GPU, the topology surgery on the host (_membrane_mesh.pyx:877-907) ---------
    def _holepunch_find_candidate_faces(self, points, eps=10.0):
        """Faces with no localisation within eps of their centre (:877-887)."""
        from .evaluation_utils import nearest_point_distance
        centres = self._vertices['position'][self.faces].mean(1)
        dist = nearest_point_distance(points, centres, _session_for(self, getattr(self, '_nw_device', 0)).aux())
        inds = np.flatnonzero(self._faces['halfedge'] != -1).astype('i4')
        return inds[dist > eps]

    def _holepunch_pair_candidate_faces(self, candidates):
        """For each candidate the opposing candidate nearest in the mean-normal plane (:898-907, the USE_C branch)."""
        candidates = np.ascontiguousarray(candidates, dtype=np.int32)
        pairs = -1 * np.ones(candidates.shape[0], dtype='i4')
        verts, faces, hes = (np.ascontiguousarray(a) for a in (self._vertices, self._faces, self._halfedges))
        if verts.dtype.itemsize != 120 or faces.dtype.itemsize != 24 or hes.dtype.itemsize != 28:
            raise RuntimeError('mesh record layouts differ from membrane_mesh_utils.h:31-65')
        if len(candidates):
            _session_for(self, getattr(self, '_nw_device', 0)).handle.call(
                'nw_holepunch_pair_candidate_faces', ctypes.c_void_p(verts.ctypes.data), ctypes.c_void_p(faces.ctypes.data),
                ctypes.c_void_p(hes.ctypes.data), len(verts), len(faces), len(hes), _lib.iptr(candidates), len(candidates), _lib.iptr(pairs))
        pair_inds = pairs != -1
        new_inds = np.cumsum(pair_inds) - 1
        return candidates[pair_inds], new_inds[pairs[pair_inds]]

    # -- block driver (_membrane_mesh.pyx:1427-1560) ---------------------------------------------------------
    def opt_conjugate_gradient(self, points, sigma, max_iter=10, step_size=1.0, weights=None, **kwargs):
        r = (self.remesh_frequency != 0) and (self.remesh_frequency <= max_iter)
        dr = (self.delaunay_remesh_frequency != 0) and (self.delaunay_remesh_frequency <= max_iter)
        if r and dr:
            rf = math.gcd(self.remesh_frequency, self.delaunay_remesh_frequency)
        elif r:
            rf = self.remesh_frequency
        elif dr:
            rf = self.delaunay_remesh_frequency
        else:
            rf = max_iter
        if r:
            initial_length = self._mean_edge_length
            if kwargs.get('minimum_edge_length', -1) < 0:
                final_length = np.clip(np.min(sigma) / 2.5, 1.0, 50.0)
            else:
                final_length = kwargs.get('minimum_edge_length')
            m = (final_length - initial_length) / (rf * np.ceil(max_iter / rf))      # linear in edge length (:1455)
        neck_first_iter = getattr(self, 'neck_first_iter', -1)

        if np.isscalar(sigma):
            s = float(sigma)                                                          # NB not inverted (:1460-1461)
        elif (len(sigma.shape) == 1) and (sigma.shape[0] == points.shape[0]):
            s = 1.0 / np.repeat(sigma, points.shape[1])
        elif (len(sigma.shape) == 2) and (sigma.shape[0] == points.shape[0]) and (sigma.shape[1] == points.shape[1]):
            s = 1.0 / sigma.ravel()
        else:
            raise ValueError(f"Sigma must be of shape ({points.shape[0]},) or ({points.shape[0]},{points.shape[1]}).")

        last_area = self.area()
        self.cg = None
        j = 0
        lams = [step_size * self.kc / 2.0, self.shrink_weight] if self.shrink_weight > 0 else [step_size * self.kc / 2.0]
        n_iter = min(max_iter, getattr(self, 'truncate_at', max_iter))
        while j < n_iter:
            self.cg = ShrinkwrapMeshConjGrad(self, points, search_k=self.search_k, search_rad=self.search_rad,
                                             shield_sigma=self._mean_edge_length / 2.0,
                                             device=getattr(self, '_nw_device', 0), comm=getattr(self, '_nw_comm', None))
            n_it = min(n_iter - j, rf)
            self.cg.search(points, lams=lams, num_iters=n_it, sigma_inv=s, weights=weights)
            j += n_it
            # host-side geometry refresh (:1524-1527)
            self._refresh_after_block()
            if dr and ((j % self.delaunay_remesh_frequency) == 0) and hasattr(self, 'punch_holes'):
                self.punch_holes(points, self.delaunay_eps)
            if r and ((j % self.remesh_frequency) == 0):
                if (neck_first_iter > 0) and (j > neck_first_iter):
                    self.remove_necks(getattr(self, 'neck_threshold_low', -1e-4), getattr(self, 'neck_threshold_high', 1e-2))
                if hasattr(self, 'remove_extra_short_edges'):
                    self.remove_extra_short_edges()
                target_length = initial_length + m * (j + 1)
                if self._host_remesh(5, target_length, 0.5, n_relax=0):
                    self.cg = None
            last_area = self.area()
        return j

    def _refresh_after_block(self):
        if hasattr(self, 'update_geometry'):          # mini-mesh
            self.update_geometry()
        else:                                         # PYME TriangleMesh property semantics
            self._face_normals_valid = 0
            self._vertex_normals_valid = 0
            self.face_normals
            self.vertex_neighbors

    def _host_remesh(self, n, target_length, l, n_relax=0):
        """Topology stays on the host: delegate to the mesh class's own remesher when it has one."""
        fn = getattr(super(), 'remesh', None)
        if fn is None:
            hook = getattr(self, 'remesh_hook', None)
            if hook is None:
                return False
            hook(self, target_length)
        else:
            fn(n, target_length, l, n_relax=n_relax)
        self._initialize_curvature_vectors()
        if hasattr(self, '_nw_session'):
            pass   # the device session is kept: points stay resident, topology is re-uploaded by the next block
        return True

    def shrink_wrap(self, points=None, sigma=None, method='conjugate_gradient', max_iter=None, **kwargs):
        """_membrane_mesh.pyx:1641-1669."""
        if method not in DESCENT_METHODS:
            print('Unknown gradient descent method. Using {}.'.format(DEFAULT_DESCENT_METHOD))
            method = DEFAULT_DESCENT_METHOD
        if max_iter is None:
            max_iter = self.max_iter
        if points is None:
            points = self._points
        if sigma is None:
            sigma = self._sigma
        self._points, self._sigma = points, sigma
        kwargs.pop('beta_1', None); kwargs.pop('beta_2', None); kwargs.pop('eps', None)
        return getattr(self, 'opt_{}'.format(method))(points=points, sigma=sigma, max_iter=max_iter,
                                                      step_size=self.step_size, **kwargs)


class MembraneMesh(ShrinkwrapMeshMixin, MiniMesh):
    """Harness mesh: mini half-edge mesh + the NanoWrap path.  ``MembraneMesh(vertices, faces, **params)`` or
    ``MembraneMesh(mesh=other)`` like the reference constructor (_membrane_mesh.pyx:79)."""

    def __init__(self, vertices=None, faces=None, mesh=None, **kwargs):
        if mesh is not None:
            vertices = np.array(mesh._vertices['position'][mesh._vertices['halfedge'] != -1]) if hasattr(mesh, '_vertices') else mesh.vertices
            faces = mesh.faces
            if hasattr(mesh, '_vertices') and not np.all(mesh._vertices['halfedge'] != -1):
                # compact deleted rows
                remap = np.cumsum(mesh._vertices['halfedge'] != -1) - 1
                faces = remap[faces]
        MiniMesh.__init__(self, vertices, faces)
        self._init_shrinkwrap(**kwargs)

    def _initialize_curvature_vectors(self):
        ShrinkwrapMeshMixin._initialize_curvature_vectors(self)

    def set_topology(self, vertices, faces):
        """Replace the mesh (used by remesh hooks in tests/bench to emulate a host remesh)."""
        keep = {k: v for k, v in self.__dict__.items() if not k.startswith('_') or k in ('_points', '_sigma', '_nw_session', '_nw_device', '_nw_comm')}
        MiniMesh.__init__(self, vertices, faces)
        self.__dict__.update(keep)
        self._initialize_curvature_vectors()
