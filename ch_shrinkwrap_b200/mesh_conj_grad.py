"""GPU-backed ``ShrinkwrapMeshConjGrad`` -- same constructor, ``search`` signature, attributes and side
effects as the reference class (``ch_shrinkwrap/mesh_conj_grad.py:19-292``), executed by libnanowrap.so.

Drop-in seam: ``MembraneMesh.opt_conjugate_gradient`` builds one of these per remesh block and calls
``search`` (``_membrane_mesh.pyx:1510-1517``).  Points are uploaded and Hilbert-sorted once per fit and the
device session is cached on the mesh object, so the per-block cost is the topology upload only.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib


class _Session:
    """Device state shared by the solver objects of one fit (one mesh object, one point cloud)."""

    def __init__(self, device=0, comm=None):
        self.handle = _lib.Handle(device)
        self.points_key = None
        self.P = 0
        self.comm = comm
        if comm is not None:
            rank, nranks, uid = comm
            self.handle.call('nw_comm_init', int(rank), int(nranks), uid)

    def aux(self):
        """A second handle on the same GPU for searches that need their own points / targets (hole-punch candidate search,
        quality metrics), so that the fit's resident localisations and topology stay untouched."""
        if getattr(self, '_aux', None) is None or self._aux.h is None:
            self._aux = _lib.Handle(self.handle.device)
        return self._aux

    def __deepcopy__(self, memo):
        return None            # device state is not copyable; a copied mesh opens its own session on first use

    def __reduce__(self):
        return (type(None), ())

    def set_points(self, points, sigma_inv, weights):
        key = (id(points), points.shape, points.dtype.str, points.__array_interface__['data'][0],
               None if np.isscalar(sigma_inv) else (id(sigma_inv), sigma_inv.__array_interface__['data'][0]),
               float(sigma_inv) if np.isscalar(sigma_inv) else None,
               None if (weights is None or np.isscalar(weights)) else (id(weights), weights.__array_interface__['data'][0]))
        if key == self.points_key:
            return
        pts = np.ascontiguousarray(points)
        P = pts.shape[0]
        if pts.dtype == np.float64:
            p32 = pts.astype(np.float32)
            if np.array_equal(p32.astype(np.float64), pts):
                pts = p32                      # exactly representable: float32 path is bit-identical
        elif pts.dtype != np.float32:
            pts = pts.astype(np.float32)
        sinv_arr, sinv_scalar = None, 1.0
        if np.isscalar(sigma_inv):
            sinv_scalar = float(sigma_inv)
        else:
            sinv_arr = _lib.as_f32(np.asarray(sigma_inv).reshape(-1))
            if sinv_arr.size != 3 * P:
                raise ValueError('sigma_inv must have 3*P entries (got %d for P=%d)' % (sinv_arr.size, P))
        w_arr = None
        if weights is not None:
            if np.isscalar(weights):
                if sinv_arr is not None or float(weights) != sinv_scalar:
                    raise NotImplementedError('scalar weights different from sigma_inv are not supported')
            else:
                w_arr = _lib.as_f32(np.asarray(weights).reshape(-1))
                if w_arr.size != 3 * P:
                    raise ValueError('weights must have 3*P entries')
        self.handle.call('nw_set_points', ctypes.c_void_p(pts.ctypes.data), int(pts.dtype == np.float64), P,
                         _lib.fptr(sinv_arr), float(sinv_scalar), _lib.fptr(w_arr))
        self.points_key = key
        self._keepalive = (points, sigma_inv, weights)
        self.P = P


def _is_vertex_t(dt):
    """True if the structured dtype is laid out like vertex_t (membrane_mesh_utils.h:57-65): the device unpacks the raw
    records by byte offset, so the fast path is only taken for exactly this layout."""
    f = dt.fields
    if dt.itemsize != 120 or f is None:
        return False
    want = {'position': (0, np.dtype(('<f4', (3,)))), 'normal': (12, np.dtype(('<f4', (3,)))), 'halfedge': (24, np.dtype('<i4')),
            'valence': (28, np.dtype('<i4')), 'neighbors': (32, np.dtype(('<i4', (20,))))}
    for name, (off, typ) in want.items():
        if name not in f or f[name][1] != off or f[name][0] != typ:
            return False
    return True


def _session_for(mesh, device=0, comm=None):
    """The device session of `mesh` (created on first use).  Normally an attribute of the mesh object; mesh classes that
    cannot take attributes (cdef classes without ``__dict__``, like the reference's ``MembraneMesh`` when it is not
    subclassed, _membrane_mesh.pyx:78) are looked up in a small module-level table instead -- the same session must come
    back for every remesh block, or each block would re-upload and re-sort all the points and leak a handle."""
    s = getattr(mesh, '_nw_session', None)
    if s is None:
        ent = _FALLBACK_SESSIONS.get(id(mesh))
        if ent is not None and ent[0] is mesh:
            s = ent[1]
            _FALLBACK_SESSIONS[id(mesh)] = _FALLBACK_SESSIONS.pop(id(mesh))      # most recently used last
    if s is None or s.handle.h is None:
        s = _Session(device, comm)
        try:
            mesh._nw_session = s
        except AttributeError:
            # the entry holds the mesh itself, so its id() cannot be recycled while the entry lives; the table is a
            # small LRU and closes what it evicts, so device memory does not pile up across many meshes
            _FALLBACK_SESSIONS.pop(id(mesh), None)
            _FALLBACK_SESSIONS[id(mesh)] = (mesh, s)
            while len(_FALLBACK_SESSIONS) > _FALLBACK_LIMIT:
                _, (_, old) = next(iter(_FALLBACK_SESSIONS.items()))
                _FALLBACK_SESSIONS.pop(next(iter(_FALLBACK_SESSIONS)))
                old.handle.close()
    return s


def release_session(mesh):
    """Free the device state of `mesh` now (otherwise it goes with the mesh object, or when the fallback table evicts it)."""
    s = getattr(mesh, '_nw_session', None)
    ent = _FALLBACK_SESSIONS.pop(id(mesh), None)
    if s is None and ent is not None and ent[0] is mesh:
        s = ent[1]
    if s is not None:
        s.handle.close()
        try:
            mesh._nw_session = None
        except AttributeError:
            pass


_FALLBACK_SESSIONS = {}      # id(mesh) -> (mesh, session), insertion order = least recently used first
_FALLBACK_LIMIT = 4


class ShrinkwrapMeshConjGrad(object):
    """See the module docstring.  Arguments as ``mesh_conj_grad.py:33``; ``sigma``, ``search_k``,
    ``search_rad``, ``shield_sigma`` and ``use_octree`` are accepted and ignored exactly like the
    reference's active path ignores them (SURVEY B.15)."""

    def __init__(self, mesh, points, sigma=None, search_k=200, search_rad=100, shield_sigma=None, use_octree=False,
                 device=0, comm=None):
        self.tests, self.ress, self.prefs = [], [], []             # conj_grad.py:37-39
        self.Lfuncs, self.Lhfuncs = ["I"], ["I"]                    # mesh_conj_grad.py:38
        self.mesh = mesh
        self._points = points
        self.sigma = sigma
        self._vertex_mask = None                                    # :44, built lazily
        self.vertices = mesh._vertices['position']                  # :46
        self.faces = mesh.faces                                     # :47
        self._vertex_neighbors = None                              # :50-54, built lazily (the device does its own lookup)
        self.M = self.vertices.shape[0]
        self.N = mesh._vertices['neighbors'].shape[1]
        self.dims = 3
        self.shape = self.vertices.shape
        self.search_k = min(search_k, points.shape[0])
        self.search_rad = max(search_rad, 1.0)
        self.loopcount = 0
        self.cpred, self.wpreds = None, None
        self._session = _session_for(mesh, device, comm)
        self._topology_uploaded = False
        self._positions_fresh = False
        self._sigma_inv, self._weights = 1.0, None
        self.f = None
        self.fs = None
        self._mask_src = None

    # -- device plumbing ---------------------------------------------------------------------------
    @property
    def points(self):
        return self._points

    @property
    def _mesh_vertex_mask(self):
        if self._vertex_mask is None:
            self._vertex_mask = self.mesh._vertices['halfedge'] != -1
        return self._vertex_mask

    @property
    def vertex_neighbors(self):
        """(M,20) neighbour vertex ids, -1 padded (mesh_conj_grad.py:50-54)."""
        if self._vertex_neighbors is None:
            nb = self.mesh._vertices['neighbors']
            n = self.mesh._halfedges['vertex'][nb]
            n[nb == -1] = -1
            self._vertex_neighbors = n
        return self._vertex_neighbors

    @property
    def _h(self):
        return self._session.handle

    def _upload_topology(self):
        mesh = self.mesh
        faces = np.ascontiguousarray(self.faces, dtype=np.int32)
        he_field = mesh._halfedges['vertex']
        verts = mesh._vertices
        nrm = mesh.vertex_normals
        if (_is_vertex_t(verts.dtype) and verts.flags.c_contiguous and isinstance(nrm, np.ndarray)
                and np.shares_memory(nrm, verts) and nrm.shape == (len(verts), 3)):
            # fast path: the records go up as they lie in memory (position, normal, halfedge, neighbors all inside); the
            # half-edge 'vertex' field is gathered out of its records by the library's upload threads
            if he_field.dtype != np.int32 or he_field.ndim != 1 or he_field.strides[0] % 4 != 0 or he_field.strides[0] < 4:
                he_field = np.ascontiguousarray(he_field, dtype=np.int32)
            self._h.call('nw_set_topology_records', ctypes.c_void_p(verts.ctypes.data), _lib.iptr(faces),
                         ctypes.c_void_p(he_field.ctypes.data), int(he_field.strides[0]),
                         int(he_field.shape[0]), int(len(verts)), int(faces.shape[0]))
        else:
            he_vertex = np.ascontiguousarray(he_field, dtype=np.int32)
            pos = _lib.as_f32(verts['position'])
            nrm = _lib.as_f32(nrm)
            nbr_he = np.ascontiguousarray(verts['neighbors'], dtype=np.int32)
            valid = np.ascontiguousarray(self._mesh_vertex_mask, dtype=np.uint8)
            self._h.call('nw_set_topology_halfedge', _lib.fptr(pos), _lib.fptr(nrm), _lib.iptr(faces), _lib.iptr(nbr_he),
                         _lib.iptr(he_vertex), int(he_vertex.shape[0]),
                         valid.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), int(pos.shape[0]), int(faces.shape[0]))
        self._topology_uploaded = True
        self._positions_fresh = True

    def _ensure_ready(self):
        self._session.set_points(self._points, self._sigma_inv, self._weights)
        if not self._topology_uploaded:
            self._upload_topology()

    # -- the hot loop ------------------------------------------------------------------------------
    def search(self, data, lams, defaults=None, num_iters=10, weights=None, sigma_inv=1.0, pos=False, last_step=True):
        """Same contract as mesh_conj_grad.py:150-292: returns the (M,3) vertex array and updates
        ``mesh._vertices['position']`` (valid rows) and the history lists."""
        if pos:
            raise NotImplementedError('pos=True (positivity constraint) is not part of the shrinkwrap path')
        if defaults is not None:
            raise NotImplementedError('explicit defaults are overwritten by the reference too (:224)')
        if type(lams) is float or np.isscalar(lams):
            lams = [float(lams)]
        if data is not self._points:
            if np.shape(data) != np.shape(self._points) or not np.array_equal(data, self._points):
                self._points = data
        # the regulariser is read from the object like the reference does (mesh_conj_grad.py:36-39,257-258)
        reg = (list(self.Lfuncs), list(self.Lhfuncs))
        if reg == (["I"], ["I"]):
            reg_mode = 0
        elif reg == (["wfunc"], ["wfunc"]):
            reg_mode = 1
        else:
            raise NotImplementedError('Lfuncs/Lhfuncs = %r: the reference\'s search() runs with ["I"] or ["wfunc"] only (its other '
                                      '1-ring operators receive a float64 array they read as float32 and fail its NaN assert)' % (reg,))
        self._sigma_inv, self._weights = sigma_inv, weights
        self._mask_src = (sigma_inv if weights is None else weights, data)   # mask is built lazily (3P bools)
        self._positions_fresh = False
        self._ensure_ready()
        if not self._positions_fresh:
            # positions may have been edited on the host since the upload (remesh happens between blocks, which builds
            # a new object, so this only matters for repeated search() calls on one object)
            posn = _lib.as_f32(self.mesh._vertices['position'])
            self._h.call('nw_set_positions', _lib.fptr(posn))
        n = int(num_iters)
        out = np.empty((self.M, 3), np.float32)
        hist = [np.zeros(max(n, 1), np.float64) for _ in range(5)]
        # the device forms the statistic in float32 like the reference, so the float32 history IS what it compared:
        # search(10) stops exactly where search(5); search(5) does
        prev = np.asarray(self.tests[-3:], dtype=np.float64)
        n_done = ctypes.c_int(0)
        lam = float(lams[0]) if len(lams) > 0 else 0.0
        self._h.call('nw_set_regulariser', reg_mode)
        self._h.call('nw_search', lam, n, int(bool(last_step)), _lib.dptr(prev) if len(prev) else None, int(len(prev)),
                     _lib.fptr(out), *[_lib.dptr(a) for a in hist], ctypes.byref(n_done))
        k = n_done.value
        self.loopcount = k
        self.tests.extend(np.float32(t) for t in hist[0][:k])
        self.ress.extend(hist[1][:k].tolist())
        self.prefs.extend(np.array([p], np.float32) for p in hist[2][:k])
        if k:
            self.cpred, self.wpreds = float(hist[3][k - 1]), [float(hist[4][k - 1])]
        self.fs = out
        self.f = out.ravel()
        dst = self.mesh._vertices['position']
        if (isinstance(dst, np.ndarray) and dst.dtype == np.float32 and dst.ndim == 2 and dst.shape == out.shape
                and dst.strides[1] == 4 and dst.strides[0] >= 12):
            # :289, written by the library row by row into the records (valid rows only)
            self._h.call('nw_get_positions_strided', ctypes.c_void_p(dst.ctypes.data), int(dst.strides[0]), 1)
        else:
            valid = self._mesh_vertex_mask
            dst[valid] = out[valid]
        self.mesh._initialize_curvature_vectors()                        # :290
        return self.fs

    # -- operators -----------------------------------------------------------------------------------
    def _ensure_weights(self):
        self._ensure_ready()
        # nw_apply_* fail if no weights exist yet: compute them at the current f like calc_w() does (:1018-1023)
        try:
            self._h.call('nw_get_weights', None, None, None, None)
        except ValueError:
            self._h.call('nw_compute_weights')

    def compute_weights(self):
        """Nearest face + weights at the mesh's current positions (_compute_weight_matrix4, :433-516)."""
        self._ensure_ready()
        self._h.call('nw_set_positions', _lib.fptr(_lib.as_f32(self.mesh._vertices['position'])))
        self._h.call('nw_compute_weights')
        return self.w

    def Afunc(self, f):
        self._ensure_weights()
        x = _lib.as_f32(np.asarray(f).reshape(-1))
        if x.size != 3 * self.M:
            raise ValueError('Afunc expects 3*M values')
        y = np.empty(3 * self._session.P, np.float32)
        self._h.call('nw_apply_A', _lib.fptr(x), _lib.fptr(y))
        return y

    def Ahfunc(self, f):
        self._ensure_weights()
        r = _lib.as_f32(np.asarray(f).reshape(-1))
        if r.size != 3 * self._session.P:
            raise ValueError('Ahfunc expects 3*P values')
        y = np.empty(3 * self.M, np.float32)
        self._h.call('nw_apply_AH', _lib.fptr(r), _lib.fptr(y))
        return y

    def point_influence(self):
        self._ensure_weights()
        pi = np.empty(self.M, np.float32)
        self._h.call('nw_point_influence', _lib.fptr(pi))
        return pi

    def surface_distance(self, points=None, return_face=False, return_closest=False, signed=False):
        """Exact distance from each point to the mesh as it stands on the device (after ``search``, the fitted surface),
        float64.  ``points=None``: the fit's own localisations, which are already resident (nothing is uploaded), in the order
        they were given.  ``return_face`` / ``return_closest`` / ``signed`` as ``evaluation_utils.surface_distance``.  This
        measures the surface itself; the fit's weights keep using the nearest face centroid (mesh_conj_grad.py:451-454)."""
        from .evaluation_utils import _surface_distances
        self._ensure_ready()
        return _surface_distances(self._h, points, self._session.P, signed, return_face, return_closest)

    def self_intersections(self, return_stats=False):
        """The intersecting face pairs of the mesh as it stands on the device (after ``search``, the fitted surface), with
        nothing uploaded: see ``evaluation_utils.self_intersections``.  The fit's own state is not touched."""
        from .evaluation_utils import _self_intersections
        self._ensure_ready()
        return _self_intersections(self._h, return_stats)

    def _ncc(self):
        self._ensure_weights()
        fd = np.empty((self.M, 3), np.float64)
        self._h.call('nw_ncc', _lib.dptr(fd))
        return fd

    def _defaults(self, idx=0):
        return self._ncc().ravel()

    def I(self, f):
        return f

    def _ring(self, name, f, ref=None):
        self._ensure_ready()
        f = _lib.as_f32(np.asarray(f).reshape(-1))
        d = np.zeros(3 * self.M, np.float32)
        if ref is None:
            self._h.call(name, _lib.fptr(f), _lib.fptr(d))
        else:
            self._h.call(name, _lib.fptr(f), _lib.fptr(_lib.as_f32(np.asarray(ref).reshape(-1))), _lib.fptr(d))
        return d

    def Lfunc(self, f):                       # mesh_conj_grad.py:590-614
        return self._ring('nw_l_func', f)

    def Lhfunc(self, f):                      # :616-638
        return self._ring('nw_lh_func', f)

    def Lfunc3(self, f):                      # :674-679  (reference geometry = self.f)
        return self._ring('nw_lw_func', f, self._current_f())

    def Lhfunc3(self, f):                     # :681-687
        return self._ring('nw_lhw_func', f, self._current_f())

    def wfunc(self, f):                       # :725-736
        self._ensure_ready()
        w = np.zeros(3 * self.M, np.float32)
        self._h.call('nw_vertex_area_weights', _lib.fptr(_lib.as_f32(self._current_f())), _lib.fptr(w))
        return np.asarray(f).reshape(-1) * w

    def _current_f(self):
        return self.f if self.f is not None else _lib.as_f32(self.mesh._vertices['position']).ravel()

    # -- read-backs (lazy: these are 3P-sized) -----------------------------------------------------------
    @property
    def mask(self):
        if self._mask_src is None:
            return None
        w_eff, data = self._mask_src
        if not np.isscalar(w_eff):
            return np.asarray(w_eff).reshape(-1) > 0               # :161
        return np.isfinite(np.asarray(data).reshape(-1))          # :164

    @property
    def res(self):
        r = np.empty(3 * self._session.P, np.float32)
        self._h.call('nw_get_res', _lib.fptr(r))
        return r

    @property
    def S(self):
        s = np.empty((3 * self.M, 3), np.float32)
        self._h.call('nw_get_S', _lib.fptr(s))
        return s

    @property
    def w(self):
        P = self._session.P
        v_idx, w = np.empty((P, 3), np.int32), np.empty((P, 3), np.float32)
        self._h.call('nw_get_weights', _lib.iptr(v_idx), _lib.fptr(w), None, None)
        return v_idx, w

    @property
    def d(self):
        P = self._session.P
        dm = np.empty(P, np.float64)
        self._h.call('nw_get_weights', None, None, _lib.dptr(dm), None)
        return np.vstack([dm, dm, dm]).T                                   # :483

    @property
    def nearest_face(self):
        P = self._session.P
        face = np.empty(P, np.int32)
        self._h.call('nw_get_weights', None, None, None, _lib.iptr(face))
        return face

    def _stop_cond(self):                                                  # :1009-1016
        if len(self.tests) < 3:
            return False
        a, b, c = self.tests[-3:]
        return (c < b) and (b < a) and (a < 1e-6)
