"""
Gaussian-process surrogate of the objective function -- the reference's ``gpso/gp_surrogate.py`` with the
GPflow/TensorFlow arithmetic replaced by the B200 library.

Kept API (reference file:line): ``GPPoint`` (:24-36), ``GPListOfPoints`` (:39-118), ``GPSurrogate`` (:121-385:
``append``, ``gp_predict``, ``gp_eval_best_ucb``, ``gp_update``, ``_gp_train``, the ``num_*`` / ``highest_*`` /
``current_training_data`` / ``gp_based_coords`` properties, optimiser (de)serialisation, ``save`` / ``from_saved``) and
``GPRSurrogate`` (:388-533, incl. ``default()``).  ``fit`` / ``predict_y`` are thin aliases named by the build brief.
``surrogate.gpflow_model`` is a :class:`pygpso_b200.gpmodel.GPR`.

Two reference conventions that parity depends on are kept verbatim: the UCB uses the *variance*
(``ucb = mean + varsigma * var``; ``score_sigma`` stores a variance, :305-308, :326) and ``predict_y`` includes the
noise variance.

Host-side change: the point list keeps a dense coordinate matrix next to the list so the duplicate test of
``append`` / ``find_by_coords`` (tolerance 1e-12, :20, :68-101) is one vectorised distance computation instead of a
Python loop over all points; order, replace-in-place and "evaluated wins" semantics are unchanged.
"""
import bisect
import itertools
import json
import logging
import os
from collections import namedtuple

import dill
import numpy as np
from scipy.special import erfcinv

from . import gpmodel
from .param_space import NORM_PARAMS_BOUNDS
from .utils import JSON_EXT, PKL_EXT, PointLabels, load_json, make_dirs

GP_TRAIN_MAX_ITER = 100
DUPLICATE_TOLERANCE = 1.0e-12


class GPPoint(namedtuple("GPPoint", ["normed_coord", "score_mu", "score_sigma", "score_ucb", "label"])):
    """One point of the surrogate: normalised coordinates, mean, variance (sic), UCB and label."""

    def __eq__(self, other):
        if not isinstance(other, tuple) or len(other) != len(self):
            return False
        return all(np.array_equal(mine, theirs) for mine, theirs in zip(self, other))

    def __ne__(self, other):
        return not self.__eq__(other)

    __hash__ = None


class GPListOfPoints(list):
    """
    List of :class:`GPPoint` whose ``append`` de-duplicates on coordinates (Euclidean distance < 1e-12, reference
    ``gp_surrogate.py:68-101``: an evaluated point is never overwritten, a GP-based one is replaced in place).

    The reference scans the whole list per lookup (O(P) per append, O(T P) per tree refresh -- the dominant cost of a
    long run once the surrogate itself is fast, SURVEY.md 8f N1).  Here the coordinates are mirrored in one array and
    indexed by a scalar projection ``w . x`` kept sorted: two points closer than the tolerance have projections closer than
    ``tol * |w|``, so a lookup is a bisection plus an exact distance check of the (almost always zero or one) points in
    that window -- same hits, same order, O(log P).  ``epoch`` changes whenever positions may have moved (generic list
    mutation); callers may cache indices against it.
    """

    @classmethod
    def from_file(cls, filename):
        if not filename.endswith(JSON_EXT):
            filename += JSON_EXT
        points = []
        for item in load_json(filename):
            item["normed_coord"] = np.array(item["normed_coord"])
            item["label"] = PointLabels[item["label"]]
            points.append(GPPoint(**item))
        return cls(points)

    def __init__(self, *args, **kwargs):
        if args:
            assert all(isinstance(it, GPPoint) for it in args[0])
        super().__init__(*args, **kwargs)
        self._reset_index()

    _uids = itertools.count(1)

    def _reset_index(self):
        self._coords = None  # [capacity, d] mirror of the coordinates of self[0:len(self)]
        self._count = 0
        self._weights = None  # projection direction
        self._keys = []       # sorted projections
        self._key_idx = []    # list positions, parallel to _keys
        self.epoch = 0
        self.uid = next(GPListOfPoints._uids)  # identity of this list for position caches (never pickled)
        self._labels = None   # positions of the evaluated / GP-based points, ascending (rebuilt lazily after generic edits)

    def __reduce__(self):
        # pickle as the plain list of points (the reference class is a bare list subclass); the index is rebuilt lazily
        return (type(self), (list(self),))

    # -- coordinate mirror + projection index ---------------------------------------------------------------------------
    def _mirror(self):
        n = len(self)
        if self._coords is None or self._count != n:
            if n == 0:
                self._coords, self._count = None, 0
                self._keys, self._key_idx = [], []
                return None
            d = np.size(self[0].normed_coord)
            cap = max(64, 2 * n)
            coords = np.empty((cap, d))
            for i, point in enumerate(self):
                coords[i] = point.normed_coord
            self._coords, self._count = coords, n
            if self._weights is None or self._weights.size != d:
                self._weights = np.random.default_rng(12345).uniform(0.5, 1.5, d)
            proj = coords[:n] @ self._weights
            order = np.argsort(proj, kind="stable")
            self._keys = proj[order].tolist()
            self._key_idx = order.tolist()
        return self._coords[: self._count]

    def _invalidate(self):
        self._coords, self._count = None, 0
        self._labels = None
        self.epoch = getattr(self, "epoch", 0) + 1

    # -- positions by label (the optimiser asks for them after every update; a scan of the list per question was a
    # visible share of a 500-evaluation run) ------------------------------------------------------------------------------
    def _label_index(self):
        if getattr(self, "_labels", None) is None:
            self._labels = {PointLabels.evaluated: [i for i, p in enumerate(self) if p.label == PointLabels.evaluated],
                            PointLabels.gp_based: [i for i, p in enumerate(self) if p.label == PointLabels.gp_based]}
        return self._labels

    def positions_with_label(self, label):
        """Ascending list positions of the points carrying ``label`` (evaluated or gp_based)."""
        return self._label_index().get(label, [])

    def _label_moved(self, position, old_label, new_label):
        if getattr(self, "_labels", None) is None or old_label == new_label:
            return
        if old_label in self._labels:
            lst = self._labels[old_label]
            at = bisect.bisect_left(lst, position)
            if at < len(lst) and lst[at] == position:
                del lst[at]
        if new_label in self._labels:
            bisect.insort(self._labels[new_label], position)

    def _window(self, coords):
        """(projection, lo, hi): the slice of the sorted projections that can hold points within the tolerance."""
        w = self._weights
        key = float(np.dot(coords, w))
        slack = DUPLICATE_TOLERANCE * float(np.sqrt(np.dot(w, w))) + 1.0e-13 * (1.0 + abs(key))
        return key, bisect.bisect_left(self._keys, key - slack), bisect.bisect_right(self._keys, key + slack)

    def _matches(self, coords):
        """Indices (ascending) of the points closer than the tolerance to ``coords``."""
        mirror = self._mirror()
        if mirror is None:
            return ()
        coords = np.asarray(coords, dtype=np.float64).reshape(-1)
        _, lo, hi = self._window(coords)
        if lo == hi:
            return ()
        cand = np.sort(np.asarray(self._key_idx[lo:hi], dtype=np.intp))
        diff = mirror[cand] - coords
        dist2 = np.einsum("ij,ij->i", diff, diff)
        return cand[np.sqrt(dist2) < DUPLICATE_TOLERANCE]

    def _index_insert(self, coords, position):
        key = float(np.dot(coords, self._weights))
        at = bisect.bisect_right(self._keys, key)
        self._keys.insert(at, key)
        self._key_idx.insert(at, position)

    def _index_remove(self, coords, position):
        key = float(np.dot(coords, self._weights))
        at = bisect.bisect_left(self._keys, key)
        while at < len(self._keys) and self._keys[at] == key:
            if self._key_idx[at] == position:
                del self._keys[at], self._key_idx[at]
                return
            at += 1
        self._invalidate()  # not found where it should be: rebuild on the next lookup

    def _store(self, position, point):
        """Replace the point at ``position`` in place (coordinates may move within the tolerance)."""
        self._label_moved(position, self[position].label, point.label)
        list.__setitem__(self, position, point)
        new = np.asarray(point.normed_coord, dtype=np.float64).reshape(-1)
        if self._coords is not None and not np.array_equal(self._coords[position], new):
            self._index_remove(self._coords[position], position)
            if self._coords is not None:
                self._coords[position] = new
                self._index_insert(new, position)

    # -- list protocol ------------------------------------------------------------------------------------------------
    def append(self, object):
        assert isinstance(object, GPPoint)
        hits = self._matches(object.normed_coord)
        if len(hits) == 0:
            n = len(self)
            super().append(object)
            if getattr(self, "_labels", None) is not None and object.label in self._labels:
                self._labels[object.label].append(n)  # positions only grow: the list stays ascending
            if self._coords is not None and self._count == n and n < self._coords.shape[0]:
                self._coords[n] = object.normed_coord
                self._count = n + 1
                self._index_insert(self._coords[n], n)
            else:
                # first point, or the mirror is full: rebuilt (with twice the capacity) by the next lookup; positions of
                # the existing points do not move, so cached indices stay valid (no epoch change)
                self._coords, self._count = None, 0
            return
        for idx in hits:
            # an evaluated point is never overwritten; a GP-based one is replaced in place
            if self[idx].label == PointLabels.evaluated:
                continue
            self._store(int(idx), object)

    def replace_at(self, positions, new_points, coords_unchanged=False):
        """Bulk replace-in-place of GP-based points whose positions are known (the re-prediction after a fit).  With
        ``coords_unchanged`` the caller guarantees that every new point carries the coordinates already stored there."""
        for position, point in zip(positions, new_points):
            assert self[position].label != PointLabels.evaluated
            if coords_unchanged:
                self._label_moved(position, self[position].label, point.label)
                list.__setitem__(self, position, point)
            else:
                self._store(int(position), point)

    def find_by_coords(self, coords):
        """First point (list order) within the tolerance of ``coords``, or None."""
        hits = self._matches(coords)
        return self[int(hits[0])] if len(hits) else None

    def index_by_coords(self, coords):
        hits = self._matches(coords)
        return int(hits[0]) if len(hits) else None

    def _mutating(name):
        def method(self, *args, **kwargs):
            self._invalidate()
            return getattr(list, name)(self, *args, **kwargs)

        method.__name__ = name
        return method

    for _name in ("__setitem__", "__delitem__", "__iadd__", "__imul__", "insert", "extend", "pop", "remove", "clear",
                  "sort", "reverse"):
        locals()[_name] = _mutating(_name)
    del _name, _mutating

    def save(self, filename):
        if not filename.endswith(JSON_EXT):
            filename += JSON_EXT
        serialised = []
        for point in self:
            item = point._asdict()
            item["normed_coord"] = np.asarray(item["normed_coord"]).tolist()
            item["label"] = item["label"].name
            serialised.append(item)
        with open(filename, "w") as handle:
            handle.write(json.dumps(serialised))


class GPSurrogate:
    """Bookkeeping of evaluated / GP-predicted points around a GP model; subclasses supply the model and its training."""

    POINTS_FILE = f"points{JSON_EXT}"
    GPR_FILE = f"GPRmodel{PKL_EXT}"
    GPR_INFO = f"GPRinfo{JSON_EXT}"

    @classmethod
    def from_saved(cls, folder):
        raise NotImplementedError

    def __init__(
        self,
        gp_kernel,
        gp_meanf=None,
        optimiser=None,
        varsigma=erfcinv(0.01),
        points=None,
        gpflow_model=None,
        backend=None,
    ):
        """
        :param gp_kernel: covariance function (``pygpso_b200.gpmodel.kernels.*``)
        :param gp_meanf: mean function (``gpmodel.mean_functions.Constant`` / ``Linear`` / ``Zero``) or None
        :param optimiser: object with ``minimize(closure, variables)``; default ``gpmodel.optimizers.Scipy()``
        :param varsigma: UCB multiplier, ``ucb = mean + varsigma * var``
        :param points: initial list of :class:`GPPoint`
        :param gpflow_model: an initialised model (only used when loading a saved surrogate)
        :param backend: compute backend; None = the CUDA library (tests inject a checker backend here)
        """
        self.gpflow_model = gpflow_model
        self.gp_varsigma = varsigma
        assert isinstance(gp_kernel, gpmodel.Kernel)
        self.gp_kernel = gp_kernel
        assert gp_meanf is None or isinstance(gp_meanf, gpmodel.MeanFunction)
        self.gp_meanf = gp_meanf
        optimiser = gpmodel.Scipy() if optimiser is None else optimiser
        assert hasattr(optimiser, "minimize")
        self.optimiser = optimiser
        self.backend = backend
        self.points = GPListOfPoints(points or list())

    # -- views on the point list --------------------------------------------------------------------------------------
    def _with_label(self, label):
        return [point for point in self.points if point.label == label]

    def _positions(self, label):
        points = self.points
        if hasattr(points, "positions_with_label"):
            return points.positions_with_label(label)
        return [i for i, point in enumerate(points) if point.label == label]

    @property
    def num_evaluated(self):
        return len(self._positions(PointLabels.evaluated))

    @property
    def num_gp_based(self):
        return len(self._positions(PointLabels.gp_based))

    @property
    def highest_score(self):
        """Evaluated point with the highest score (first one on ties), or None."""
        best = None
        for point in self.points:
            if point.label == PointLabels.evaluated and (best is None or point.score_mu > best.score_mu):
                best = point
        return best

    @property
    def highest_ucb(self):
        """GP-based point with the highest UCB (first one on ties), or None."""
        best = None
        for point in self.points:
            if point.label == PointLabels.gp_based and (best is None or point.score_ucb > best.score_ucb):
                best = point
        return best

    @property
    def current_training_data(self):
        evaluated = self._with_label(PointLabels.evaluated)
        x = np.array([point.normed_coord for point in evaluated])
        y = np.array([point.score_mu for point in evaluated])
        return x, y

    @property
    def gp_based_coords(self):
        return np.array([point.normed_coord for point in self._with_label(PointLabels.gp_based)])

    # -- to be provided by the concrete surrogate ---------------------------------------------------------------------
    def _gp_train(self, x, y):
        raise NotImplementedError

    def save(self, folder):
        raise NotImplementedError

    # -- data ---------------------------------------------------------------------------------------------------------
    def append(self, coords, scores):
        """Add objective evaluations (normalised ``coords[n,d]``, ``scores[n]``) as training points."""
        assert coords.ndim == 2
        assert scores.ndim == 1
        assert coords.shape[0] == scores.shape[0]
        for idx in range(coords.shape[0]):
            self.points.append(
                GPPoint(
                    normed_coord=coords[idx, :],
                    score_mu=scores[idx],
                    score_sigma=0.0,
                    score_ucb=0.0,
                    label=PointLabels.evaluated,
                )
            )

    # -- prediction ---------------------------------------------------------------------------------------------------
    def _require_model(self):
        assert isinstance(self.gpflow_model, gpmodel.GPModel), "train the surrogate (gp_update / _gp_train) first"
        return self.gpflow_model

    def predict_y(self, normed_coords):
        """Posterior mean and variance (noise included), both ``[M,1]``; alias of ``gpflow_model.predict_y``."""
        return self._require_model().predict_y(normed_coords)

    def gp_predict(self, normed_coords):
        """Predict at ``normed_coords[M,d]`` and store one GP-based point per row (duplicates replace in place)."""
        mean, var = self._require_model().predict_y(normed_coords)
        mean = np.asarray(mean).reshape(-1)
        var = np.asarray(var).reshape(-1)
        for idx in range(normed_coords.shape[0]):
            self.points.append(
                GPPoint(
                    normed_coord=normed_coords[idx, :],
                    score_mu=float(mean[idx]),
                    score_sigma=float(var[idx]),
                    score_ucb=float(mean[idx] + self.gp_varsigma * var[idx]),
                    label=PointLabels.gp_based,
                )
            )

    def gp_eval_best_ucb(self, normed_coords):
        """(mean, var, ucb) of the candidate with the highest ``mean + varsigma*var`` (first one on ties).  With a process
        group every rank passes the same candidates and scores its own contiguous shard of them."""
        model = self._require_model()
        scorer = self._sharded_scorer()
        if scorer is not None:
            _, mean, var, ucb = scorer.ucb_argmax_full(np.ascontiguousarray(normed_coords, dtype=np.float64), self.gp_varsigma)
        else:
            _, mean, var, ucb = model.ucb_argmax(normed_coords, self.gp_varsigma)
        return mean, var, ucb

    def gp_eval_best_ucb_in_leaf(self, leaf, depth):
        """
        ``gp_eval_best_ucb(leaf.grow(depth))`` without the round trip through the host: the leaf-centre batch is
        generated on the device and scored in place (reference optimisation.py:379-381).  With a process group every rank
        generates and scores its own slice of the batch.
        """
        model = self._require_model()
        scorer = self._sharded_scorer()
        if scorer is not None:
            _, mean, var, ucb = scorer.grow_ucb_argmax(leaf.bounds_array(), depth, self.gp_varsigma)
        else:
            _, mean, var, ucb = model.grow_ucb_argmax(leaf.bounds_array(), depth, self.gp_varsigma)
        return mean, var, ucb

    # -- multi-GPU (SURVEY.md 8e): one process per GPU, every rank holds a replica of the surrogate ------------------------
    group = None

    def _world(self):
        from .distributed import _rank_world

        return _rank_world(None if self.group in (None, True) else self.group) if self.group is not None else (0, 1)

    def _sharded_scorer(self):
        """``ShardedScorer`` over this rank's session when the surrogate was given a process group of more than one rank."""
        if self.group is None or self._world()[1] == 1:
            return None
        from .distributed import ShardedScorer

        session = self._require_model()._session
        scorer = getattr(self, "_scorer", None)
        if scorer is None or scorer.session is not session:
            scorer = self._scorer = ShardedScorer(session, None if self.group is True else self.group)
        return scorer

    def _broadcast_fit(self):
        """After a fit: rank 0 factorises, its state (scaled inputs, alpha, L^-1, hyper-parameters) is broadcast once and
        imported by the other ranks, so every rank scores with bit-identical factors."""
        scorer = self._sharded_scorer()
        if scorer is None:
            return
        model = self._require_model()
        n, d = model.data[0].shape
        if scorer.rank == 0:
            model._ensure_factor()
        scorer.broadcast_fit(n, d, src=0)
        if scorer.rank != 0:
            model._factor_key = model._theta().tobytes()  # the imported factor belongs to the hyper-parameters in force

    def gp_update(self):
        """Re-train on all evaluated points, then refresh every GP-based point with the new posterior."""
        x_train, y_train = self.current_training_data
        if logging.getLogger().isEnabledFor(logging.DEBUG):
            logging.debug(f"Retraining GPR with x data: {x_train}; y data: {y_train}")
        self._gp_train(x=x_train, y=y_train[:, np.newaxis])
        # gp_predict(gp_based_coords) of the reference (gp_surrogate.py:341-342) with the positions carried along: one
        # batched predict_y, then every GP-based point is replaced in place without the per-row duplicate search
        positions = list(self._positions(PointLabels.gp_based))
        if positions:
            coords = np.array([self.points[i].normed_coord for i in positions])
            mean, var = self._require_model().predict_y(coords)
            mean = np.asarray(mean).reshape(-1)
            var = np.asarray(var).reshape(-1)
            ucb = mean + self.gp_varsigma * var
            self.points.replace_at(
                positions,
                (
                    GPPoint(normed_coord=coords[k], score_mu=float(mean[k]), score_sigma=float(var[k]), score_ucb=float(ucb[k]),
                            label=PointLabels.gp_based)
                    for k in range(len(positions))
                ),
                coords_unchanged=True,
            )

    def fit(self, x=None, y=None):
        """Alias: train on (x, y[:,None]) or, without arguments, on the evaluated points."""
        if x is None:
            x, y = self.current_training_data
            y = y[:, np.newaxis]
        return self._gp_train(x=x, y=y)

    # -- optimiser (de)serialisation ----------------------------------------------------------------------------------
    def _serialise_optimiser(self):
        name = self.optimiser.__class__.__name__
        if name == "Scipy":
            return tuple([name])
        raise ValueError(f"{name} not currently supported.")

    @staticmethod
    def _deserialse_optimiser(from_json):
        if from_json[0] == "Scipy":
            return gpmodel.Scipy()
        raise ValueError(f"{from_json[0]} not currently supported.")


class GPRSurrogate(GPSurrogate):
    """Surrogate on exact GP regression with a Gaussian likelihood."""

    def __init__(
        self,
        gp_kernel,
        gp_meanf=None,
        optimiser=None,
        varsigma=erfcinv(0.01),
        gauss_likelihood_sigma=1.0e-3,
        points=None,
        gpflow_model=None,
        backend=None,
        n_restarts=1,
        group=None,
        restart_maxiter=50,
        restart_seed=20240517,
    ):
        """
        :param gauss_likelihood_sigma: initial noise *variance* of the Gaussian likelihood (normalised units)
        :param n_restarts: multi-start restarts of every hyper-parameter fit.  Restart 0 is the reference's own fit (warm
            start, the optimiser's full budget), so 1 reproduces the reference trajectory; restarts i > 0 start at
            ``u + N(0,1)`` in unconstrained space with ``restart_maxiter`` iterations; the smallest -LML wins
        :param group: ``True`` (default process group) or a ``torch.distributed`` group: one process per GPU, every rank
            builds the same surrogate and calls the same methods (SPMD).  Restarts are dealt round-robin over the ranks,
            the fitted state is broadcast once per fit, candidates / leaf batches are sharded over the ranks
        """
        super().__init__(
            gp_kernel=gp_kernel,
            gp_meanf=gp_meanf,
            optimiser=optimiser,
            varsigma=varsigma,
            points=points,
            gpflow_model=gpflow_model,
            backend=backend,
        )
        self.gp_lik_sigma = gauss_likelihood_sigma
        assert int(n_restarts) >= 1
        self.n_restarts = int(n_restarts)
        self.group = group
        self.restart_maxiter = restart_maxiter
        self.restart_seed = restart_seed

    @classmethod
    def default(cls, backend=None, **kwargs):
        """Matern-5/2 with lengthscale 0.25, unit variance, constant mean 0, noise variance 1e-3, SciPy L-BFGS-B."""
        return cls(
            gp_kernel=gpmodel.Matern52(lengthscales=np.sum(NORM_PARAMS_BOUNDS) * 0.25, variance=1.0),
            gp_meanf=gpmodel.Constant(0.0),
            optimiser=gpmodel.Scipy(),
            varsigma=erfcinv(0.01),
            gauss_likelihood_sigma=1.0e-3,
            points=None,
            gpflow_model=None,
            backend=backend,
            **kwargs,
        )

    def _gp_train(self, x, y):
        assert x.shape[0] == y.shape[0]
        assert x.ndim == 2 and y.ndim == 2
        if self.gpflow_model is None:
            self.gpflow_model = gpmodel.GPR(
                data=(x, y),
                kernel=self.gp_kernel,
                mean_function=self.gp_meanf,
                noise_variance=self.gp_lik_sigma,
                backend=self.backend,
            )
        else:
            self.gpflow_model.data = (x, y)  # hyper-parameters warm-start from the previous optimum
        model = self.gpflow_model
        rank, world = self._world()
        if self.n_restarts == 1 and world == 1:
            return self.optimiser.minimize(model.training_loss, model.trainable_variables)
        # restart 0 = the reference's fit with the surrogate's own optimiser (on the rank that owns it), the other restarts
        # through SciPy L-BFGS-B from perturbed starts; (-LML*, u*) of every restart is gathered and the winner installed on
        # every rank -- identical hyper-parameters everywhere, bit for bit
        from .distributed import multistart_fit

        result = multistart_fit(self, model, self.n_restarts, None if self.group in (None, True) else self.group,
                                seed=self.restart_seed, maxiter=self.restart_maxiter)
        self._broadcast_fit()
        return result

    # -- persistence: same file names and JSON keys as the reference (:505-533 / :436-482) -----------------------------
    def save(self, folder):
        make_dirs(folder)
        self.points.save(filename=os.path.join(folder, self.POINTS_FILE))
        model = self._require_model()
        params = {key: np.asarray(p).copy() for key, p in gpmodel.parameter_dict(model).items()}
        with open(os.path.join(folder, self.GPR_FILE), "wb") as handle:
            dill.dump(params, handle)
        meanf = model.mean_function
        is_sum = isinstance(model.kernel, gpmodel.Combination)  # a Sum or a Product
        periodic = isinstance(model.kernel, gpmodel.Periodic)
        leaf = model.kernel.base_kernel if periodic else model.kernel
        linear = isinstance(leaf, gpmodel.LinearKernel)  # no lengthscales: the shape saved is the variance's
        save_info = {
            "gpr_kernel": model.kernel.__class__.__name__,
            "gpr_kernel_shape": [] if is_sum else (leaf.variance if linear else leaf.lengthscales).shape.as_list(),
            "gpr_meanf": meanf.__class__.__name__,
            "gpr_meanf_shape": meanf.parameters[0].shape.as_list() if meanf.parameters else [],
            "gp_varsigma": self.gp_varsigma,
            "gp_likelihood": self.gp_lik_sigma,
            "optimiser": self._serialise_optimiser(),
        }
        if is_sum:  # component (factor) families and lengthscale shapes, in order
            # a periodic term: ["Periodic", base lengthscale shape, base family, period shape]; a Linear term: ["Linear", variance shape]
            save_info["gpr_kernel_components"] = [
                ["Periodic", k.base_kernel.lengthscales.shape.as_list(), k.base_kernel.__class__.__name__, k.period.shape.as_list()]
                if isinstance(k, gpmodel.Periodic) else ["Linear", k.variance.shape.as_list()] if isinstance(k, gpmodel.LinearKernel)
                else [k.__class__.__name__, k.lengthscales.shape.as_list()]
                for k in model.kernel.kernels]
        if periodic:  # base family and the shape of the period; gpr_kernel_shape is the base lengthscales'
            save_info["gpr_kernel_periodic"] = [leaf.__class__.__name__, model.kernel.period.shape.as_list()]
        leaves = model.kernel.kernels if is_sum else [model.kernel]
        if any(gpmodel._active_dims_given(k.active_dims) for k in leaves):  # per leaf: its resolved columns, or null
            save_info["gpr_kernel_active_dims"] = [
                list(dims) if gpmodel._active_dims_given(k.active_dims) else None for k, dims in zip(leaves, model._leaf_dims)]
        with open(os.path.join(folder, self.GPR_INFO), "w") as handle:
            handle.write(json.dumps(save_info))

    @classmethod
    def from_saved(cls, folder, backend=None, **kwargs):
        points = GPListOfPoints.from_file(os.path.join(folder, cls.POINTS_FILE))
        evaluated = [point for point in points if point.label == PointLabels.evaluated]
        x = np.array([point.normed_coord for point in evaluated])
        y = np.array([point.score_mu for point in evaluated])[:, np.newaxis]

        info = load_json(os.path.join(folder, cls.GPR_INFO))
        assert hasattr(gpmodel.kernels, info["gpr_kernel"])
        if info["gpr_kernel"] in ("Sum", "Product"):  # multiple_assign restores every component's parameters below
            def component(entry):
                if entry[0] == "Periodic":
                    return gpmodel.kernels.Periodic(getattr(gpmodel.kernels, entry[2])(lengthscales=np.ones(entry[1])),
                                                    period=np.ones(entry[3]))
                if entry[0] == "Linear":
                    return gpmodel.kernels.Linear(variance=np.ones(entry[1]))
                return getattr(gpmodel.kernels, entry[0])(lengthscales=np.ones(entry[1]))
            gp_kernel = getattr(gpmodel.kernels, info["gpr_kernel"])([component(e) for e in info["gpr_kernel_components"]])
        elif info["gpr_kernel"] == "Periodic":
            base, period_shape = info["gpr_kernel_periodic"]
            gp_kernel = gpmodel.kernels.Periodic(getattr(gpmodel.kernels, base)(lengthscales=np.ones(info["gpr_kernel_shape"])),
                                                 period=np.ones(period_shape))
        elif info["gpr_kernel"] == "Linear":
            gp_kernel = gpmodel.kernels.Linear(variance=np.ones(info["gpr_kernel_shape"]))
        else:
            gp_kernel = getattr(gpmodel.kernels, info["gpr_kernel"])(lengthscales=np.ones(info["gpr_kernel_shape"]))
        if "gpr_kernel_active_dims" in info:
            leaves = gp_kernel.kernels if isinstance(gp_kernel, gpmodel.Combination) else [gp_kernel]
            for k, dims in zip(leaves, info["gpr_kernel_active_dims"]):
                k.active_dims = dims
        assert hasattr(gpmodel.mean_functions, info["gpr_meanf"])
        meanf_cls = getattr(gpmodel.mean_functions, info["gpr_meanf"])
        if meanf_cls is gpmodel.Constant:
            gp_meanf = meanf_cls(np.zeros(info["gpr_meanf_shape"]))
        elif meanf_cls is gpmodel.Linear:  # gpr_meanf_shape is the shape of A, [d, 1]; multiple_assign restores A and b below
            gp_meanf = meanf_cls(np.zeros(info["gpr_meanf_shape"]), np.zeros(1))
        else:
            gp_meanf = meanf_cls()
        optimiser = cls._deserialse_optimiser(info["optimiser"])

        model = gpmodel.GPR(
            data=(x, y), kernel=gp_kernel, mean_function=gp_meanf, noise_variance=info["gp_likelihood"], backend=backend
        )
        with open(os.path.join(folder, cls.GPR_FILE), "rb") as handle:
            params = dill.load(handle)
        gpmodel.multiple_assign(model, params)
        return cls(
            gp_kernel=gp_kernel,
            gp_meanf=gp_meanf,
            optimiser=optimiser,
            gauss_likelihood_sigma=info["gp_likelihood"],
            varsigma=info["gp_varsigma"],
            points=points,
            gpflow_model=model,
            backend=backend,
            **kwargs,
        )
