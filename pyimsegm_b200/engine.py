"""
Device-resident driver of the SLIC -> descriptors -> GraphCut hot path.

Everything here is plumbing: torch tensors are used purely as device-memory containers and every computation is
a call into ``libimsegm_b200.so`` through the C-ABI (``include/imsegm_b200.h``).  No torch op touches the data
path.  The numpy-facing modules (``superpixels``, ``descriptors``, ``graph_cuts``, ``pipelines``, ``tiled``, ``texture``) are thin
wrappers over this class, and :meth:`Engine.call` is the only way they reach the library.
"""
import ctypes as C

import numpy as np

from . import _lib

_DOUBLE_P = C.POINTER(C.c_double)
FLAG_BITS = {'mean': 1, 'std': 2, 'energy': 4}
#: initial capacity of a device edge table, in edges per node of a 4-connected label map (twice that for a 6-connected volume)
EDGE_CAP_PER_NODE = 8
#: edge_type -> (metric, spatial) of isb_gc_energies; only 'model' and 'spatial' are spatially normalised
#: (reference graph_cuts.py:646)
EDGE_MODES = {'': (0, 0), 'model': (1, 1), 'model_lT': (1, 0), 'model_l1': (2, 0), 'model_l2': (3, 0), 'spatial': (0, 1)}


def flag_bits(flags):
    """(bit mask, number of statistics) of a list of FLAG_BITS names"""
    bits = 0
    for f in flags:
        bits |= FLAG_BITS[f]
    return bits, bin(bits).count('1')


def dtype_code(dtype):
    """C-ABI element type code of a numpy or torch dtype"""
    name = str(dtype)
    return _lib.DTYPE_CODES[name[len('torch.'):] if name.startswith('torch.') else np.dtype(dtype).name]


def edge_capacity(nodes, ndim=2):
    """rows of a device edge table over ``nodes`` labels of a ``ndim``-D label map, first attempt: EDGE_CAP_PER_NODE per node
    (twice as many in 3-D)"""
    return max(64, EDGE_CAP_PER_NODE * (ndim - 1) * int(nodes))


def grown_edge_capacity(cap):
    """rows of the next attempt after a table of ``cap`` rows overflowed.  An overflowed table reports cap + 1 edges and no
    kernel reads it, so the retry computes the same whatever the growth factor."""
    return 4 * int(cap)


def gaussian_half_kernel(sigma, truncate=4.0):
    """half of scipy.ndimage's normalised 1-D Gaussian: [w0, w1 .. wr], radius r = int(truncate * sigma + 0.5)"""
    radius = int(truncate * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    phi = phi / phi.sum()
    return np.ascontiguousarray(phi[radius:], dtype=np.float64), radius


def regular_grid_steps(shape, n_points):
    """(start, step) per axis of skimage.util.regular_grid for an array of ``shape`` and ``n_points`` seeds"""
    shape = np.asarray(shape)
    ndim = len(shape)
    rank = np.argsort(np.argsort(shape))
    dims = np.sort(shape)
    space = float(np.prod(shape))
    if space <= n_points:
        return [(0, 1)] * ndim
    steps = np.full(ndim, (space / n_points) ** (1.0 / ndim))
    if (dims < steps).any():
        for d in range(ndim):
            steps[d] = dims[d]
            space = float(np.prod(dims[d + 1:]))
            steps[d + 1:] = (space / n_points) ** (1.0 / (ndim - d - 1))
            if (dims >= steps).all():
                break
    starts = (steps // 2).astype(int)
    steps = np.round(steps).astype(int)
    pairs = [(int(a), int(b)) for a, b in zip(starts, steps)]
    return [pairs[i] for i in rank]


def slic_seed_grid(H, W, n_segments):
    (_, _), (sy, ty), (sx, tx) = regular_grid_steps((1, H, W), n_segments)
    gy, gx = np.meshgrid(np.arange(sy, H, ty), np.arange(sx, W, tx), indexing='ij')
    seeds = np.stack([gy.ravel(), gx.ravel()], axis=1).astype(np.float64)
    return np.ascontiguousarray(seeds), int(ty), int(tx)


def slic_seed_grid3d(shape, n_segments):
    """seeds (z, y, x) of skimage's regular grid over a volume and the per-axis steps"""
    (sz, tz), (sy, ty), (sx, tx) = regular_grid_steps(shape, n_segments)
    gz, gy, gx = np.meshgrid(np.arange(sz, shape[0], tz), np.arange(sy, shape[1], ty), np.arange(sx, shape[2], tx), indexing='ij')
    seeds = np.stack([gz.ravel(), gy.ravel(), gx.ravel()], axis=1).astype(np.float64)
    return np.ascontiguousarray(seeds), (int(tz), int(ty), int(tx))


class Engine(object):
    """owns the device buffers for one image shape at a time and sequences the C-ABI calls on the current stream"""

    def __init__(self, device=None):
        self.torch = _lib.require_cuda()
        self.lib = _lib.lib()
        self.device = self.torch.device('cuda', self.torch.cuda.current_device() if device is None else device)
        self._bufs = {}
        self._fns = {name[len('isb_'):]: getattr(self.lib, name) for name in _lib.SIGNATURES}

    # -- C-ABI calls -----------------------------------------------------------------------------------------------
    def call(self, name, *args):
        """``isb_<name>(*args, stream)`` on the CURRENT stream (read at every call: graph capture and the side stream switch it),
        raising on an error status.  A torch tensor passes as its device pointer, a (float64) numpy array as a pointer to its
        data, anything else as it is (the argtypes of ``_lib.SIGNATURES`` convert numbers and take a struct by reference)."""
        tensor = self.torch.Tensor
        _lib.check(self._fns[name](*[a.data_ptr() if isinstance(a, tensor) else a.ctypes.data_as(_DOUBLE_P) if isinstance(a, np.ndarray)
                                     else a for a in args], self.torch.cuda.current_stream().cuda_stream))

    def query(self, name, *args):
        """value of the host-side C-ABI function ``isb_<name>(*args)`` (workspace sizes, launch counter)"""
        return self._fns[name](*args)

    def workspace(self, name, query, *args):
        """cached byte buffer ``name`` of the size ``isb_<query>(*args)`` asks for; returns (buffer, bytes)"""
        wsb = self._fns[query](*args)
        return self.buf(name, (wsb,), self.torch.uint8), wsb

    # -- memory helpers ------------------------------------------------------------------------------------------
    def buf(self, name, shape, dtype):
        """cached device buffer (grown on demand, never shrunk)"""
        torch = self.torch
        if torch.cuda.current_device() != self.device.index:
            # the C-ABI calls launch on the CURRENT device's stream: an engine must only be driven with its own device current
            raise RuntimeError('Engine of cuda:%d used while cuda:%d is the current device' % (self.device.index, torch.cuda.current_device()))
        shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        n = int(np.prod(shape)) if shape else 1
        cur = self._bufs.get(name)
        if cur is None or cur.dtype != dtype or cur.numel() < n:
            if cur is not None and getattr(self, 'graphs_captured', 0):
                # a captured CUDA graph may hold the address of the old block: keep it alive instead of returning it to the allocator
                self.__dict__.setdefault('_retired', []).append(cur)
            cur = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._bufs[name] = cur
        return cur[:n].view(shape)

    #: host arrays at least this large that are NOT page-locked go through the staged upload below
    STAGE_MIN_BYTES = 4 << 20
    STAGE_CHUNK = 4 << 20
    STAGE_SLOTS = 8

    def to_device(self, arr, name=None):
        """host ndarray -> device tensor through the current stream (pinned sources copy asynchronously; large pageable sources
        are staged, see :meth:`_staged_upload`)"""
        torch = self.torch
        arr = np.ascontiguousarray(arr)
        src = torch.from_numpy(arr)
        if name is None:
            return src.to(self.device, non_blocking=True)
        dst = self.buf(name, arr.shape, src.dtype)
        if arr.nbytes >= self.STAGE_MIN_BYTES and not src.is_pinned():
            self._staged_upload(dst, arr)
        else:
            dst.copy_(src, non_blocking=True)
        return dst

    def _staged_upload(self, dst, arr):
        """upload of a large PAGEABLE array (what a caller of the numpy API normally holds): the driver would bounce it through
        its own small staging buffer at a fraction of the PCIe rate.  Here worker threads copy 4 MB chunks into a ring of pinned
        buffers (numpy releases the GIL while copying) and every chunk is sent by an asynchronous DMA as soon as it is complete, so
        the host copies overlap the transfers."""
        torch = self.torch
        if getattr(self, '_stage', None) is None:
            from concurrent.futures import ThreadPoolExecutor
            slots = [torch.empty(self.STAGE_CHUNK, dtype=torch.uint8, pin_memory=True) for _ in range(self.STAGE_SLOTS)]
            self._stage = (slots, [t.numpy() for t in slots], [torch.cuda.Event() for _ in slots], [False] * len(slots),
                           ThreadPoolExecutor(self.STAGE_SLOTS))
        slots, views, events, used, pool = self._stage
        src = arr.reshape(-1).view(np.uint8)
        out = dst.view(torch.uint8).reshape(-1)
        n, ch = src.shape[0], self.STAGE_CHUNK
        nchunks = (n + ch - 1) // ch

        def fill(slot, lo, hi):
            np.copyto(views[slot][:hi - lo], src[lo:hi])

        def submit(c):
            slot = c % len(slots)
            if used[slot]:
                events[slot].synchronize()      # the DMA that last read this slot has finished
            return pool.submit(fill, slot, c * ch, min(n, (c + 1) * ch))

        futs = {c: submit(c) for c in range(min(len(slots), nchunks))}
        for c in range(nchunks):
            slot = c % len(slots)
            futs.pop(c).result()
            lo, hi = c * ch, min(n, (c + 1) * ch)
            out[lo:hi].copy_(slots[slot][:hi - lo], non_blocking=True)
            events[slot].record()
            used[slot] = True
            if c + len(slots) < nchunks:
                futs[c + len(slots)] = submit(c + len(slots))

    def const_device(self, arr, name):
        """small host array that rarely changes between calls (seed grid, pairwise table, filter taps): every distinct content gets
        its OWN device tensor, uploaded once and never overwritten -- no copy in steady state, and a captured CUDA graph that read
        one of them keeps reading the right values whatever other configurations run in between"""
        import hashlib
        arr = np.ascontiguousarray(arr)
        key = (name, arr.shape, arr.dtype.str, hashlib.blake2b(arr.tobytes(), digest_size=16).digest())
        cache = self.__dict__.setdefault('_consts', {})
        hit = cache.get(key)
        if hit is not None:
            return hit
        if self.torch.cuda.is_current_stream_capturing():
            raise RuntimeError('constant %r is new while a CUDA graph is being captured' % name)
        dst = self.torch.from_numpy(arr).to(self.device)
        cache[key] = dst
        return dst

    def pinned_empty(self, shape, dtype):
        """pinned host tensor (torch's caching host allocator recycles the blocks once the result is dropped)"""
        return self.torch.empty(tuple(shape), dtype=dtype, pin_memory=True)

    def to_host(self, t, sync=True):
        out = self.pinned_empty(t.shape, t.dtype)
        out.copy_(t, non_blocking=True)
        if sync:
            self.torch.cuda.current_stream().synchronize()
        return out.numpy()

    def download(self, tensors):
        """copies of device tensors into pinned host tensors, queued on the current stream; returns (host tensors, an event recorded
        after the copies) -- the caller synchronises on the event when it needs the data"""
        hosts = []
        for t in tensors:
            h = self.pinned_empty(t.shape, t.dtype)
            h.copy_(t, non_blocking=True)
            hosts.append(h)
        event = self.torch.cuda.Event()
        event.record()
        return hosts, event

    def side_stream(self):
        """a second CUDA stream of this engine (copies that may overlap the kernels of the main stream)"""
        if getattr(self, '_side', None) is None:
            self._side = self.torch.cuda.Stream(device=self.device)
        return self._side

    # -- (i) SLIC -------------------------------------------------------------------------------------------------
    @staticmethod
    def slic_setup(H, W, n_segments, sigma):
        """host-side set-up of the whole-image and the banded SLIC: (half Gaussian kernel, its radius, seed grid [n, 2], step_y,
        step_x, step)"""
        w_half, radius = gaussian_half_kernel(sigma) if sigma > 0 else (np.ones(1), 0)
        seeds, ty, tx = slic_seed_grid(H, W, n_segments)
        return w_half, radius, seeds, ty, tx, float(max(1, ty, tx))

    def connectivity(self, km, n_segments, min_size_factor=0.5, max_size_factor=3):
        """connectivity pass over a k-means label map [H, W]; returns (labels int32 [H, W], n_labels device int32[1])"""
        H, W = int(km.shape[0]), int(km.shape[1])
        segment_size = H * W / n_segments
        min_size, max_size = int(min_size_factor * segment_size), int(max_size_factor * segment_size)
        cws, cwsb = self.workspace('ws_conn', 'connectivity_workspace_bytes', H, W)
        out = self.buf('labels', (H, W), self.torch.int32)
        n_labels = self.buf('n_labels', (1,), self.torch.int32)
        self.call('enforce_connectivity', km, H, W, min_size, max_size, out, n_labels, cws, cwsb)
        return out, n_labels

    def slic(self, d_img, n_segments, compactness, sigma=1.0, max_iter=10, enforce_connectivity=True,
             min_size_factor=0.5, max_size_factor=3, slic_zero=False, rescale=True):
        """device SLIC on a [H,W,C] device tensor; returns (labels int32 [H,W] device, n_labels device int32[1] or None)"""
        torch = self.torch
        H, W = int(d_img.shape[0]), int(d_img.shape[1])
        Cn = 1 if d_img.dim() == 2 else int(d_img.shape[2])
        w_half, radius, seeds, ty, tx, step = self.slic_setup(H, W, n_segments, sigma)
        lab = self.buf('lab', (3, H, W), torch.float64)
        mm = self.buf('minmax', (4,), torch.float64)
        self.call('slic_prepare', d_img, dtype_code(d_img.dtype), H, W, Cn, w_half, radius, 1.0 / compactness, int(bool(rescale)), lab, mm)
        n_seeds = len(seeds)
        d_seeds = self.const_device(seeds, 'seeds')
        ws, wsb = self.workspace('ws_kmeans', 'slic_kmeans_workspace_bytes', H, W, n_seeds, ty, tx)
        km = self.buf('labels_km', (H, W), torch.int32)
        self.call('slic_kmeans', lab, H, W, d_seeds, n_seeds, ty, tx, step, int(max_iter), int(bool(slic_zero)), km, None, ws, wsb)
        if not enforce_connectivity:
            return km, None
        return self.connectivity(km, n_segments, min_size_factor, max_size_factor)

    def slic3d(self, d_vol, n_segments, compactness, spacing=(1, 1, 1), sigma=1.0, max_iter=10, enforce_connectivity=True,
               min_size_factor=0.5, max_size_factor=3):
        """device SLIC of a single-channel volume [D, H, W] (csrc/slic3d.cu); returns (labels int32 [D,H,W], n_labels or None)"""
        torch = self.torch
        D, H, W = (int(v) for v in d_vol.shape)
        spacing = np.ascontiguousarray(spacing, dtype=np.float64)
        halves = []
        for axis, sig in enumerate(np.array([sigma, sigma, sigma], dtype=np.float64) / spacing):
            w_half, radius = gaussian_half_kernel(sig) if sigma > 0 else (np.ones(1), 0)
            halves += [self.to_device(w_half, 'slic3d_w%d' % axis), radius]
        tmp = self.buf('slic3d_tmp', (D, H, W), torch.float64)
        scaled = self.buf('slic3d_vol', (D, H, W), torch.float64)
        self.call('slic3d_prepare', d_vol, dtype_code(d_vol.dtype), D, H, W, *halves, 1.0 / compactness, tmp, scaled)
        seeds, steps = slic_seed_grid3d((D, H, W), n_segments)
        n_seeds = len(seeds)
        d_seeds = self.to_device(seeds, 'seeds3d')
        ws, wsb = self.workspace('ws_kmeans3d', 'slic3d_kmeans_workspace_bytes', D, H, W, n_seeds)
        km = self.buf('labels_km3d', (D, H, W), torch.int32)
        self.call('slic3d_kmeans', scaled, D, H, W, d_seeds, n_seeds, steps[0], steps[1], steps[2], float(max(steps)), spacing,
                  int(max_iter), km, ws, wsb)
        if not enforce_connectivity:
            return km, None
        segment_size = D * H * W / n_segments
        min_size, max_size = int(min_size_factor * segment_size), int(max_size_factor * segment_size)
        cws, cwsb = self.workspace('ws_conn3d', 'connectivity3d_workspace_bytes', D, H, W, max(max_size, 1))
        out = self.buf('labels3d', (D, H, W), torch.int32)
        n_labels = self.buf('n_labels', (1,), torch.int32)
        self.call('enforce_connectivity3d', km, D, H, W, min_size, max_size, out, n_labels, cws, cwsb)
        return out, n_labels

    def centroids3d(self, d_seg, nb):
        """centres (z, y, x) [nb, 3] of the labels of a device label volume"""
        nb = int(nb)
        centres = self.buf('centres3d', (nb, 3), self.torch.float64)
        cws = self.buf('ws_centres3d', (4 * nb,), self.torch.int64)
        self.call('centroids_3d', d_seg, *d_seg.shape, nb, centres, cws, 32 * nb)
        return centres

    def slic_label_bound(self, H, W, n_segments, min_size_factor=0.5):
        """upper bound on the number of labels after connectivity enforcement (each kept label has >= min_size px)"""
        min_size = max(1, int(min_size_factor * (H * W / n_segments)))
        return H * W // min_size + 1

    # -- (ii) descriptors -----------------------------------------------------------------------------------------
    def segment_stats(self, d_img, d_seg, nb, flags, feat=None, col0=0, want_centres=False, want_counts=False):
        """colour statistics (+centroids) of a [H,W,3] device image over labels [H,W] int32 in [0, nb)"""
        torch = self.torch
        H, W = int(d_seg.shape[0]), int(d_seg.shape[1])
        nb = int(nb)
        bits, n = flag_bits(flags)
        if feat is None and n:
            feat = self.buf('feat', (nb, 3 * n), torch.float64)
        ld = int(feat.shape[1]) if feat is not None else 0
        centres = self.buf('centres', (nb, 2), torch.float64) if want_centres else None
        counts = self.buf('counts', (nb,), torch.int32) if want_counts else None
        ws, wsb = self.workspace('ws_stats', 'segment_stats_workspace_bytes', nb)
        self.call('segment_stats_2d', d_img, 0 if d_img is None else dtype_code(d_img.dtype), d_seg, H, W, nb, bits, feat, ld, int(col0),
                  centres, counts, ws, wsb)
        return feat, centres, counts

    # -- (iii) graph, energies, alpha-expansion ---------------------------------------------------------------------
    def adjacency(self, d_seg, nb, cap=None):
        """unique 4-connected (6-connected in a volume) label pairs of a device label map;
        returns (edges int32 [cap,2] device, n_edges device int32[1], cap)"""
        torch = self.torch
        nb = int(nb)
        cap = edge_capacity(nb, d_seg.dim()) if cap is None else int(cap)
        ws, wsb = self.workspace('ws_adj', 'adjacency_workspace_bytes', nb, cap)
        edges = self.buf('edges', (cap, 2), torch.int32)
        n_edges = self.buf('n_edges', (1,), torch.int32)
        self.call('adjacency_edges' if d_seg.dim() == 2 else 'adjacency_edges_3d', d_seg, *d_seg.shape, nb, edges, cap, n_edges, ws, wsb)
        return edges, n_edges, cap

    def gc_energies(self, d_proba, d_edges, E, d_n_edges, d_centres, edge_mode, edge_cost, pairwise, d_n_nodes=None):
        torch = self.torch
        N, K, E = int(d_proba.shape[0]), int(d_proba.shape[1]), int(E)
        d_pw = self.const_device(np.ascontiguousarray(pairwise, dtype=np.float64), 'pairwise')
        unary = self.buf('unary', (N, K), torch.float64)
        edge_w = self.buf('edge_w', (max(E, 1),), torch.float64)
        unary_i = self.buf('unary_i', (N, K), torch.int32)
        edge_wi = self.buf('edge_wi', (max(E, 1),), torch.int32)
        smooth_i = self.buf('smooth_i', (K, K), torch.int32)
        ws, wsb = self.workspace('ws_energy', 'gc_energies_workspace_bytes', N, K, E)
        self.call('gc_energies', d_proba, N, d_n_nodes, K, d_edges, E, d_n_edges, d_centres, int(edge_mode[0]), int(edge_mode[1]),
                  float(edge_cost), d_pw, unary, edge_w, unary_i, edge_wi, smooth_i, ws, wsb)
        return unary, edge_w, unary_i, edge_wi, smooth_i

    def alpha_expansion(self, N, K, E, d_n_edges, d_edges, edge_wi, unary_i, smooth_i, n_iter=-1, init_labels=None,
                        d_n_nodes=None):
        torch = self.torch
        N, K, E = int(N), int(K), int(E)
        labels = self.buf('gc_labels', (N,), torch.int32)
        if init_labels is None:
            self.call('fill_i32', labels, N, 0)
        else:
            labels.copy_(init_labels)  # device-to-device memcpy of a caller-supplied labeling
        energy = self.buf('gc_energy', (1,), torch.int64)
        stats = self.buf('gc_stats', (8,), torch.int32)
        ws, wsb = self.workspace('ws_gc', 'alpha_expansion_workspace_bytes', N, K, E)
        self.call('alpha_expansion', N, d_n_nodes, K, E, d_n_edges, d_edges, edge_wi, unary_i, smooth_i, int(n_iter), labels, energy,
                  stats, ws, wsb)
        return labels, energy, stats

    def graph_cut(self, d_proba, d_edges, E, d_n_edges, d_centres, edge_mode, edge_cost, pairwise, d_n_nodes=None):
        """energies of the superpixel graph [N = d_proba rows, K classes] and the alpha-expansion over them (asynchronous);
        returns (labels [N] int32, unary [N, K], edge weights [E]) on the device"""
        unary, edge_w, unary_i, edge_wi, smooth_i = self.gc_energies(d_proba, d_edges, E, d_n_edges, d_centres, edge_mode, edge_cost,
                                                                     pairwise, d_n_nodes=d_n_nodes)
        labels, _, _ = self.alpha_expansion(d_proba.shape[0], d_proba.shape[1], E, d_n_edges, d_edges, edge_wi, unary_i, smooth_i, -1,
                                            d_n_nodes=d_n_nodes)
        return labels, unary, edge_w

    def gmm_fit_predict(self, d_feat, K, n_init, max_iter, use_scaler=True, seed=0, d_n=None, init_labels=None, tol=1e-3,
                        reg_covar=1e-6):
        """device class model: returns (proba [N,K] device, params device vector; see isb_gmm_fit_predict)"""
        torch = self.torch
        N, D, K, n_init = int(d_feat.shape[0]), int(d_feat.shape[1]), int(K), int(n_init)
        ld = int(d_feat.stride(0))
        proba = self.buf('proba', (N, K), torch.float64)
        params = self.buf('gmm_params', (self.query('gmm_params_len', D, K),), torch.float64)
        ws, wsb = self.workspace('ws_gmm', 'gmm_workspace_bytes', N, D, K, n_init)
        d_init = None
        if init_labels is not None:
            d_init = self.to_device(np.ascontiguousarray(init_labels, dtype=np.int32), 'gmm_init')
        self.call('gmm_fit_predict', d_feat, N, D, ld, d_n, K, n_init, int(max_iter), float(tol), float(reg_covar), int(bool(use_scaler)),
                  int(seed), d_init, proba, params, ws, wsb)
        return proba, params

    def gmm_predict(self, d_feat, d_model, K, d_n=None):
        """class probabilities [N, K] (the cached 'proba' buffer) of the features [N, D] under a GIVEN model, the device vector
        packed by :class:`graph_cuts.DeviceClassModel` (see isb_gmm_predict); ``d_n``: device row count, rows beyond it untouched"""
        N, D, K = int(d_feat.shape[0]), int(d_feat.shape[1]), int(K)
        proba = self.buf('proba', (N, K), self.torch.float64)
        ws, wsb = self.workspace('ws_gmm_predict', 'gmm_predict_workspace_bytes', N, D, K)
        self.call('gmm_predict', d_feat, N, D, int(d_feat.stride(0)), d_n, K, d_model, proba, ws, wsb)
        return proba

    def gather(self, d_seg, lut_i=None, lut_p=None, out_i=None):
        """segm = lut_i[seg] (into ``out_i`` or the cached 'segm') and segm_soft = lut_p[seg] over a device label map [H, W]"""
        torch = self.torch
        H, W = int(d_seg.shape[0]), int(d_seg.shape[1])
        if out_i is None and lut_i is not None:
            out_i = self.buf('segm', (H, W), torch.int32)
        K = int(lut_p.shape[1]) if lut_p is not None else 0
        out_p = self.buf('segm_soft', (H, W, K), torch.float64) if lut_p is not None else None
        self.call('gather', d_seg, H * W, lut_i, lut_p, K, out_i, out_p)
        return out_i, out_p


_ENGINES = {}


def get_engine(device=None):
    """one engine per device (buffers are cached inside)"""
    torch = _lib.require_cuda()
    idx = torch.cuda.current_device() if device is None else int(device)
    if idx not in _ENGINES:
        _ENGINES[idx] = Engine(idx)
    return _ENGINES[idx]
