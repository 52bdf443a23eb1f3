"""Multi-object / multi-frame pose estimation over the GPUs of one box (SURVEY.md §8f N3): pure replicas.

The reference's dataset drivers are strictly sequential — `run_ycb_video.py:116-121` / `run_linemod.py:119-123` loop over
objects, call `est.reset_object(...)` once per object and then `est.register(...)` frame after frame on one GPU.  The
frames of one object are independent, so here every GPU holds its own estimator (own fp_ctx: weights, mesh copy, frame,
workspaces, CUDA graphs) and a worker thread per GPU pulls frames from a shared queue.  ctypes releases the GIL around
every libfpose call, so the workers run concurrently inside ONE process (the reference's process model); nothing is
exchanged between GPUs.

    pool = ReplicaPool(range(torch.cuda.device_count()))
    for ob_id, mesh in meshes.items():                      # run_ycb_video.py:99-118
        pool.reset_object(mesh.vertices, mesh.vertex_normals, mesh=mesh, symmetry_tfs=sym[ob_id])
        poses = pool.register_many(frames_of[ob_id])        # [(K, rgb, depth, ob_mask), ...] -> [(4,4), ...] in order
"""
import queue
import threading

import torch

from .engine import Engine
from .estimater import FoundationPose, PoseRefinePredictor, ScorePredictor


class _Worker(threading.Thread):
    def __init__(self, device, jobs, state_dicts, cfg, cluster_symmetries=False, make_estimator=None):
        super().__init__(daemon=True)
        self.device, self.jobs, self.state_dicts, self.cfg = int(device), jobs, state_dicts, cfg
        self.cluster_symmetries = cluster_symmetries
        self.make_estimator = make_estimator
        self.est = None
        self.ready = threading.Event()
        self.error = None

    def _build(self, model_pts, model_normals, mesh, symmetry_tfs):
        if self.make_estimator is not None:
            self.est = self.make_estimator(self.device, model_pts, model_normals, mesh, symmetry_tfs)
            return
        eng = Engine()
        refiner = PoseRefinePredictor(engine=eng, state_dict=self.state_dicts.get("refine"), cfg=self.cfg.get("refine"))
        scorer = ScorePredictor(engine=eng, state_dict=self.state_dicts.get("score"), cfg=self.cfg.get("score"))
        # the rotation grid is built at construction (estimater.py:40-41): without `cluster_symmetries` it is the full
        # 252-pose grid for every object, as in the reference's drivers, whose placeholder Box has no symmetry
        self.est = FoundationPose(model_pts=model_pts, model_normals=model_normals,
                                  symmetry_tfs=symmetry_tfs if self.cluster_symmetries else None, mesh=mesh, scorer=scorer, refiner=refiner)
        if not self.cluster_symmetries:
            self.est.reset_object(model_pts, model_normals, symmetry_tfs=symmetry_tfs, mesh=mesh)

    def run(self):
        # a custom estimator's device id may be a label only (the host-side test double): select it only if it exists
        try:
            if self.make_estimator is None or self.device < torch.cuda.device_count():
                torch.cuda.set_device(self.device)
        except Exception as ex:  # no such device: every job fails with this, instead of the caller waiting forever
            self.error = ex
        while True:
            job = self.jobs.get()
            if job is None:
                return
            kind, payload, done = job
            try:
                if self.error is not None:
                    raise self.error
                if kind == "reset":
                    model_pts, model_normals, mesh, symmetry_tfs = payload
                    if self.est is None:
                        self._build(model_pts, model_normals, mesh, symmetry_tfs)
                    else:
                        self.est.reset_object(model_pts, model_normals, symmetry_tfs=symmetry_tfs, mesh=mesh)
                        if self.cluster_symmetries:
                            self.est.make_rotation_grid(min_n_views=40, inplane_step=60)
                    done(None)
                else:
                    K, rgb, depth, mask, iteration = payload
                    done(self.est.register(K=K, rgb=rgb, depth=depth, ob_mask=mask, iteration=iteration))
            except Exception as ex:  # surfaced by the pool
                done(ex)


class ReplicaPool:
    """One estimator per GPU, fed from queues.  `state_dicts` = {"refine": ..., "score": ...} (None: checkpoints found
    the reference's way, else the seeded stand-ins), `cfg` likewise.  `cluster_symmetries`: False keeps the reference
    drivers' behaviour — `reset_object` (estimater.py:43-85) stores an object's symmetry transforms but the 252 start
    poses built at construction are NOT re-clustered under them; True thins the start poses per object (fewer hypotheses
    for symmetric objects, same pose up to the symmetry group).  `make_estimator(device, model_pts, model_normals, mesh,
    symmetry_tfs)`: build each replica's estimator some other way (an object with `reset_object` / `register`; the
    scheduling tests use it with a host-side double)."""

    def __init__(self, device_ids, state_dicts=None, cfg=None, cluster_symmetries=False, make_estimator=None):
        self.device_ids = [int(d) for d in device_ids]
        self._private = [queue.Queue() for _ in self.device_ids]  # per-replica commands (reset_object)
        self.workers = []
        for d, q in zip(self.device_ids, self._private):
            w = _Worker(d, q, state_dicts or {}, cfg or {}, cluster_symmetries, make_estimator)
            w.start()
            self.workers.append(w)

    def close(self):
        for q in self._private:
            q.put(None)
        for w in self.workers:
            w.join(timeout=30)

    def reset_object(self, model_pts, model_normals, symmetry_tfs=None, mesh=None):
        """estimater.py:43-85 on every replica (each GPU gets its own copy of the mesh)."""
        results, ev = [], threading.Semaphore(0)

        def done(r):
            results.append(r)
            ev.release()

        for q in self._private:
            q.put(("reset", (model_pts, model_normals, mesh, symmetry_tfs), done))
        for _ in self._private:
            ev.acquire()
        for r in results:
            if isinstance(r, Exception):
                raise r

    def register_many(self, frames, iteration=5):
        """frames: sequence of (K, rgb, depth, ob_mask).  Returns the (4,4) poses in input order.  Dynamic
        scheduling: every replica takes the next unprocessed frame as soon as it is free."""
        frames = list(frames)
        out = [None] * len(frames)
        lock = threading.Lock()
        cursor = [0]
        finished = threading.Semaphore(0)

        def feed(q):
            # one pump per replica: hands its worker the next frame, waits for the result, repeats
            while True:
                with lock:
                    i = cursor[0]
                    cursor[0] += 1
                if i >= len(frames):
                    finished.release()
                    return
                got = threading.Event()

                def done(r, i=i, got=got):
                    out[i] = r
                    got.set()

                K, rgb, depth, mask = frames[i]
                q.put(("register", (K, rgb, depth, mask, iteration), done))
                got.wait()

        pumps = [threading.Thread(target=feed, args=(q,), daemon=True) for q in self._private]
        for p in pumps:
            p.start()
        for _ in pumps:
            finished.acquire()
        for r in out:
            if isinstance(r, Exception):
                raise r
        return out
