#!/usr/bin/env python
"""bench.py -- frames/s of the OpenVSLAM hot path on synthetic streams (BASELINE.json configs).

  --config 4 (default)  configs[3]: 1920x960 equirectangular, 4000 kp/frame: extract + robust::brute_force_match +
                        projection::match_frame_and_landmarks (20k landmarks) + pose_optimizer + local_bundle_adjuster
                        (50 free + 10 fixed keyframes, 20k landmarks, ~100k observations).  The metric's configuration.
  --config 2            configs[1]: 752x480 mono (EuRoC shape), 1000 kp: extract + projection::match_current_and_last_frames
  --config 3            configs[2]: 1241x376 stereo pairs (KITTI shape), 2000 kp: extract L + R, stereo::compute, pose_optimizer
  --config 5            configs[4]: 1920x1080 perspective, 2000 kp, the config-4 pipeline, one stream per GPU

One "step" = --frames-per-step frames (default 8) through the hot path on each of the --streams independent camera streams
of a GPU (every stream owns its handles, CUDA streams and host thread); --warmup W (at least 3) untimed steps precede the
--steps K timed ones.  Two measurements per run, over the SAME calls:
  value  every input already resident in HBM when the timed region starts (frames, BA graph): ovs_extract_device,
         ovs_robust_brute_force_match_device, ovs_frame_index_create_device, ovs_local_ba_prepare_device / run / fetch_device.
         The whole path is inside the timed region -- graph preparation, greedy replays, Levenberg loop -- only the
         host<->device copies of the inputs / results are not.
  e2e    the host-buffer C-ABI entry points a reference caller would use, every host<->device copy inside the timed region.
`--impl reference` times the CPU oracle (the restated reference; the real one cannot be built here, see DESIGN.md) on the
same workload with all usable host cores, as independent streams.  Prints ONE JSON line on rank 0.
`--dump-outputs DIR` writes what the value leg returned for the last frame of each camera stream as DIR/stream<k>_<name>.npy
(float32 / float64); the inputs depend only on the arguments, so two builds can be compared output for output."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/sec extract+match+local-BA @1920x960 4000kp"
CONFIGS = {
    2: dict(W=752, H=480, NKP=1000, model="perspective", stereo=False, ba=False, streams=8,
            name="configs[1]: 752x480 mono stream (EuRoC shape), 1000 kp/frame, extract + match::projection::match_current_and_last_frames"),
    3: dict(W=1241, H=376, NKP=2000, model="perspective", stereo=True, ba=False, streams=8,
            name="configs[2]: 1241x376 stereo pairs (KITTI shape), 2000 kp/frame, extract L+R + match::stereo::compute + pose_optimizer"),
    4: dict(W=1920, H=960, NKP=4000, model="equirectangular", stereo=False, ba=True, streams=8,
            name="configs[3]: 1920x960 equirectangular stream, 4000 kp/frame, extract + brute-force match + projection match (20k landmarks) "
                 "+ pose_optimizer + local_bundle_adjuster (50+10 KF / 20k landmarks / ~100k obs)"),
    5: dict(W=1920, H=1080, NKP=2000, model="perspective", stereo=False, ba=True, streams=1,
            name="configs[4]: 1920x1080 perspective stream, 2000 kp/frame, one stream per GPU, extract + brute-force match + projection match "
                 "(20k landmarks) + pose_optimizer + local_bundle_adjuster (50+10 KF / 20k landmarks)"),
}
K_FREE, K_FIXED, N_LM = 50, 10, 20000
N_PROJ_LM = 20000          # landmarks projected into the frame by match_frame_and_landmarks


def host_cores():
    """CPU cores this process may actually use: the cgroup CPU quota when there is one (the GPU boxes show 128 logical
    CPUs but cap the container at 16 cores), else the affinity mask / cpu count."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def max_over_ranks(elapsed, device, world):
    """MAX over ranks of a per-rank elapsed time (the contract's timing rule)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([elapsed], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def aggregate_value(frames_per_rank, elapsed, world):
    """Whole-job throughput: every rank processed `frames_per_rank` frames of its own streams (weak scaling)."""
    return world * frames_per_rank / elapsed


# ------------------------------------------------------------------------------ synthetic workload
def make_workload(cfg, seed, ring_frames):
    """Seeded frames (a ring larger than L2), the per-frame matcher inputs and the optimiser problems of one rank."""
    from openvslam_b200 import synth
    W, H, NKP = cfg["W"], cfg["H"], cfg["NKP"]
    nbase = 6
    base = [synth.frame(W, H, seed=seed * 100 + i) for i in range(nbase)]
    shift = 37 if cfg["model"] == "equirectangular" else 3
    frames, shifts = [], []
    for i in range(ring_frames):
        s = shift * (i // nbase)
        frames.append(np.ascontiguousarray(np.roll(base[i % nbase], s, axis=1)))   # equirectangular yaw / small pan
        shifts.append(s)
    wl = dict(frames=frames, shifts=shifts, nbase=nbase)
    if cfg["stereo"]:
        wl["disparity"] = 24
        wl["frames_right"] = [np.ascontiguousarray(np.roll(f, -wl["disparity"], axis=1)) for f in frames]
    if cfg["ba"]:
        wl["ba"] = synth.ba_problem(K_FREE, K_FIXED, N_LM, model=cfg["model"], seed=seed + 4)
    wl["pose"] = synth.pose_problem(NKP, model=cfg["model"], seed=seed + 3, stereo=cfg["stereo"])
    return wl


def make_landmark_sets(cfg, wl, ext):
    """Per base frame: the landmarks a tracker would project into it.  Config 4 / 5: 20k local map points -- one per keypoint
    of the frame (reprojection within sigma 2 px of it, predicted level = its octave, descriptor = the keypoint's with a few
    bits flipped) and, as in a real local map, a majority that project into the image but were not detected in this frame
    (uniform positions, unrelated descriptors).  Config 2: the 'last frame' of match_current_and_last_frames -- its keypoints."""
    rng = np.random.default_rng(17)
    sets = []
    W, H = cfg["W"], cfg["H"]
    for b in range(wl["nbase"]):
        kps, desc = ext.extract(wl["frames"][b])
        n = len(kps)
        xy = np.stack([kps["x"], kps["y"]], 1).astype(np.float32) + rng.normal(0, 2.0, (n, 2)).astype(np.float32)
        d = desc.copy()
        flip = rng.integers(0, 256, d.shape, dtype=np.uint8) & rng.integers(0, 256, d.shape, dtype=np.uint8) & rng.integers(0, 256, d.shape, dtype=np.uint8)
        d ^= flip & rng.integers(0, 256, d.shape, dtype=np.uint8)
        level = kps["octave"].astype(np.int32); angle = kps["angle"].astype(np.float32)
        if cfg["ba"]:
            extra = max(0, N_PROJ_LM - n)
            xy = np.concatenate([xy, np.stack([rng.uniform(0, W, extra), rng.uniform(0, H, extra)], 1).astype(np.float32)])
            d = np.concatenate([d, rng.integers(0, 256, (extra, 32), dtype=np.uint8)])
            level = np.concatenate([level, rng.integers(0, 8, extra).astype(np.int32)]); angle = np.concatenate([angle, rng.uniform(0, 360, extra).astype(np.float32)])
            perm = rng.permutation(len(xy))              # the map's own order, not the frame's
            xy, d, level, angle = xy[perm], d[perm], level[perm], angle[perm]
        sets.append(dict(xy=np.ascontiguousarray(xy), level=np.ascontiguousarray(level), desc=np.ascontiguousarray(d), angle=np.ascontiguousarray(angle)))
    return sets


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu,power.draw"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]

        def col(i):
            out = []
            for r in self.rows:
                try:
                    out.append(float(r[i]))
                except (ValueError, IndexError):
                    pass
            return out
        util, power = col(6), col(7)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "gpu_util_pct_median": float(np.median(util)) if util else None,
                "power_w_median": float(np.median(power)) if power else None}


STAGES = ("extract", "brute_force_match", "projection_match", "stereo_match", "pose_optimizer", "local_ba")


class CameraStream:
    """One camera stream: its own extractor / matcher / optimiser handles (each with a private CUDA stream), as the
    reference owns them per tracking / mapping thread.  Streams are independent, so S of them per GPU is the same
    weak-scaling unit as one stream per rank."""

    def __init__(self, cfg, sid, local, dev, d_frames, h_frames, d_frames_r, h_frames_r, wl, lmsets, ring, spec, cluster, spec2=0, graphs=False):
        import torch
        from openvslam_b200 import feature, match, optimize, _lib
        self.cfg, self.sid, self.ring, self.wl, self.lmsets = cfg, sid, ring, wl, lmsets
        W, H, NKP = cfg["W"], cfg["H"], cfg["NKP"]
        self.L = _lib.lib()
        self._lib = _lib
        self.dev = dev
        self.ext = feature.orb_extractor(feature.orb_params(max_num_keypts=NKP), device=local)
        self.ext_r = feature.orb_extractor(feature.orb_params(max_num_keypts=NKP), device=local) if cfg["stereo"] else None
        self.mt = match.robust(lowe_ratio=0.75, device=local)
        self.pj = match.projection(device=local)
        self.st = match.stereo(device=local) if cfg["stereo"] else None
        self.po = optimize.pose_optimizer(device=local)
        pose = wl["pose"]
        self.pcam = optimize.camera(**pose["cam"])
        self.grid = match.camera_grid(0, W, 0, H)
        self.sf = np.array([1.2 ** i for i in range(8)], np.float32)
        self.d_frames, self.h_frames, self.d_frames_r, self.h_frames_r = d_frames, h_frames, d_frames_r, h_frames_r
        self.cap = self.L.ovs_extractor_max_keypoints(self.ext._h)
        self.d_kps = torch.zeros((2, self.cap, 28), dtype=torch.uint8, device=dev)
        self.d_desc = torch.zeros((2, self.cap, 32), dtype=torch.uint8, device=dev)
        if cfg["stereo"]:
            self.d_kps_r = torch.zeros((self.cap, 28), dtype=torch.uint8, device=dev)
            self.d_desc_r = torch.zeros((self.cap, 32), dtype=torch.uint8, device=dev)
        if cfg["ba"]:
            ba = wl["ba"]
            self.cam = optimize.camera(**ba["cam"])
            self.ba_args = (ba["poses"], ba["fixed"], ba["points"], ba["obs_kf"], ba["obs_lm"], ba["obs_xy"], None, ba["inv_sigma_sq"])
            self.lba = optimize.local_bundle_adjuster(device=local)
            self.pba = optimize.prepared_local_ba.__new__(optimize.prepared_local_ba)
            optimize._optimizer_handle.__init__(self.pba, local)
            self.lba.set_speculation(spec); self.pba.set_speculation(spec)
            self.lba.set_second_batch(spec2); self.pba.set_second_batch(spec2)
            if graphs:
                self.lba.set_graphs(True); self.pba.set_graphs(True)
            self.lba.set_cluster_width(cluster); self.pba.set_cluster_width(cluster)
            # the BA graph resident in HBM (value leg): what a caller that keeps its map on the GPU would hold
            self.d_ba = {k: torch.from_numpy(np.ascontiguousarray(ba[k], dt)).to(dev) for k, dt in
                         (("poses", np.float64), ("fixed", np.uint8), ("points", np.float64), ("obs_kf", np.int32), ("obs_lm", np.int32),
                          ("obs_xy", np.float32), ("inv_sigma_sq", np.float32))}
            self.d_ba_out = (torch.zeros_like(self.d_ba["poses"]), torch.zeros_like(self.d_ba["points"]),
                             torch.zeros(len(ba["obs_kf"]), dtype=torch.uint8, device=dev))
        self.n_prev, self.prev_desc, self.prev_kps = 0, None, None
        self.last = {}                                 # host-side results of the last step_device frame (outputs())
        self.stage_ms = {"device": np.zeros(len(STAGES)), "host": np.zeros(len(STAGES))}
        self.reset()

    def reset(self):
        self.st_dev = {"match_us": 0.0, "ext_us": np.zeros(8), "ba_us": 0.0, "pose_us": 0.0, "frames": 0, "match_calls": 0,
                       "solver_us": 0.0, "schur_us": 0.0, "co_observations": 0, "solver_launches": 0, "solver_trials": 0, "reduced_dim": 0, "ba_trials": 0, "ba_iterations": 0}
        for v in self.stage_ms.values():
            v[:] = 0

    # -- matcher inputs of frame i (landmarks follow the frame's pan)
    def _landmarks(self, i):
        s = self.lmsets[i % self.wl["nbase"]]
        xy = s["xy"].copy()
        xy[:, 0] = (xy[:, 0] + self.wl["shifts"][i]) % self.cfg["W"]
        return s, xy

    def _common_tail(self, leg, fidx, n, i, t):
        """projection match of frame i on the frame index `fidx` -> the matched landmark of every keypoint (-1: none); t = stage clock list."""
        cfg = self.cfg
        s, xy = self._landmarks(i)
        if cfg["ba"]:
            _, matched = self.pj.match_frame_and_landmarks(fidx, self.sf, xy, None, s["level"], s["desc"], None, None, 5.0)
        else:
            _, matched = self.pj.match_current_and_last_frames(fidx, self.sf, 8, np.ones(len(xy), np.uint8), xy, None, s["level"], s["angle"], s["desc"], None, 20.0)
        fidx.close()
        t.append(time.perf_counter())
        return matched

    def step_device(self, i):
        i = (i + 11 * self.sid) % self.ring            # streams walk the shared frame ring at different offsets
        cfg, L, sd = self.cfg, self.L, self.st_dev
        W, H = cfg["W"], cfg["H"]
        cur = i & 1
        t = [time.perf_counter()]
        n = self.ext.extract_device(self.d_frames[i].data_ptr(), W, H, W, self.d_kps[cur].data_ptr(), self.d_desc[cur].data_ptr(), self.cap)
        sd["ext_us"] += np.array(list(self.ext.last_timings_us().values()))
        if cfg["stereo"]:
            nr = self.ext_r.extract_device(self.d_frames_r[i].data_ptr(), W, H, W, self.d_kps_r.data_ptr(), self.d_desc_r.data_ptr(), self.cap)
        t.append(time.perf_counter())
        pose = self.wl["pose"]
        last = {"frame": i, "num_keypoints": n}
        if cfg["stereo"]:
            last["num_keypoints_right"] = nr
            # stereo::compute takes the keypoint / descriptor arrays of both images (the API of the reference): they come to the
            # host once, the pyramids stay on the device
            kl = self.d_kps[cur][:n].cpu().numpy().view(self._kp_dtype()).reshape(-1); dl = self.d_desc[cur][:n].cpu().numpy()
            kr = self.d_kps_r[:nr].cpu().numpy().view(self._kp_dtype()).reshape(-1); dr = self.d_desc_r[:nr].cpu().numpy()
            last["stereo_x_right"], last["stereo_depth"], _ = self.st.compute(self.ext, self.ext_r, kl, dl, kr, dr, pose["cam"]["focal_x_baseline"],
                                                                              pose["cam"]["focal_x_baseline"] / pose["cam"]["fx"])
            t.append(time.perf_counter())
            stages = ["extract", "stereo_match"]
        else:
            stages = ["extract"]
            if cfg["ba"]:
                if self.n_prev:
                    last["brute_force_matches"] = self.mt.brute_force_match_device(self.d_desc[cur].data_ptr(), n, self.d_desc[cur ^ 1].data_ptr(), self.n_prev)
                    sd["match_us"] += self.mt.last_kernel_us(); sd["match_calls"] += 1
                self.n_prev = n
                t.append(time.perf_counter()); stages.append("brute_force_match")
            from openvslam_b200 import match
            fidx = match.frame_index.from_device(self.pj, n, self.d_kps[cur].data_ptr(), self.d_desc[cur].data_ptr(), self.grid)
            last["projection_matches"] = self._common_tail("device", fidx, n, i, t); stages.append("projection_match")
        xr = pose["obs_xr"] if cfg["stereo"] else None
        _, last["pose"], last["pose_outliers"], pst = self.po.optimize(self.pcam, not cfg["stereo"], pose["pts_w"], pose["obs_xy"], xr, pose["inv_sigma_sq"],
                                                                        pose["poses"][0])
        self.last = last
        sd["pose_us"] += pst["device_us"]
        t.append(time.perf_counter()); stages.append("pose_optimizer")
        if cfg["ba"]:
            from openvslam_b200 import optimize
            d, ba = self.d_ba, self.wl["ba"]
            optimize.prepared_local_ba.from_device(self.cam, True, len(ba["poses"]), len(ba["points"]), len(ba["obs_kf"]), d["poses"].data_ptr(),
                                                   d["fixed"].data_ptr(), d["points"].data_ptr(), d["obs_kf"].data_ptr(), d["obs_lm"].data_ptr(),
                                                   d["obs_xy"].data_ptr(), None, d["inv_sigma_sq"].data_ptr(), handle=self.pba)
            bst = self.pba.run()
            o = self.d_ba_out
            self._lib.check(L.ovs_local_ba_fetch_device(self.pba._h, C.c_void_p(o[0].data_ptr()), C.c_void_p(o[1].data_ptr()), C.c_void_p(o[2].data_ptr())))
            sd["ba_us"] += bst["device_us"]; sd["solver_us"] += bst["solver_us"]; sd["solver_launches"] += bst["solver_launches"]
            sd["solver_trials"] += bst["solver_trials"]; sd["reduced_dim"] = bst["reduced_dim"]
            sd["schur_us"] += bst["schur_us"]; sd["co_observations"] = bst["co_observations"]
            sd["ba_trials"] += bst["num_trials"]; sd["ba_iterations"] += bst["num_iterations"]
            t.append(time.perf_counter()); stages.append("local_ba")
        sd["frames"] += 1
        self._clock("device", stages, t)
        return n

    def step_host(self, i):
        i = (i + 11 * self.sid) % self.ring
        cfg = self.cfg
        pose = self.wl["pose"]
        from openvslam_b200 import match
        t = [time.perf_counter()]
        kps, desc = self.ext.extract(self.h_frames[i])
        if cfg["stereo"]:
            kps_r, desc_r = self.ext_r.extract(self.h_frames_r[i])
        t.append(time.perf_counter())
        if cfg["stereo"]:
            self.st.compute(self.ext, self.ext_r, kps, desc, kps_r, desc_r, pose["cam"]["focal_x_baseline"], pose["cam"]["focal_x_baseline"] / pose["cam"]["fx"])
            t.append(time.perf_counter())
            stages = ["extract", "stereo_match"]
        else:
            stages = ["extract"]
            if cfg["ba"]:
                if self.prev_desc is not None:
                    self.mt.brute_force_match(desc, self.prev_desc)
                self.prev_desc = desc
                t.append(time.perf_counter()); stages.append("brute_force_match")
            fidx = match.frame_index(self.pj, kps["x"], kps["y"], kps["octave"], kps["angle"], None, desc, self.grid)
            self._common_tail("host", fidx, len(kps), i, t); stages.append("projection_match")
        xr = pose["obs_xr"] if cfg["stereo"] else None
        self.po.optimize(self.pcam, not cfg["stereo"], pose["pts_w"], pose["obs_xy"], xr, pose["inv_sigma_sq"], pose["poses"][0])
        t.append(time.perf_counter()); stages.append("pose_optimizer")
        if cfg["ba"]:
            self.lba.optimize(self.cam, True, *self.ba_args)
            t.append(time.perf_counter()); stages.append("local_ba")
        self._clock("host", stages, t)
        return len(kps)

    def _clock(self, leg, stages, t):
        acc = self.stage_ms[leg]
        for k, name in enumerate(stages):
            acc[STAGES.index(name)] += (t[k + 1] - t[k]) * 1e3

    @staticmethod
    def _kp_dtype():
        from openvslam_b200 import feature
        return feature.KEYPOINT_DTYPE

    def outputs(self):
        """What the last step_device frame handed its caller, as float32 / float64 host arrays by name: keypoints (x, y, size,
        angle, response, octave per row), descriptors (one byte value per column), match results (-1: no match), the optimised
        pose and its outlier flags, and the local BA's poses, points and outlier flags."""
        last = dict(self.last)
        cur = last.pop("frame") & 1

        def keypoints(d_kps, d_desc, n):
            k = d_kps[:n].cpu().numpy().view(self._kp_dtype()).reshape(-1)
            return (np.stack([k[f].astype(np.float32) for f in ("x", "y", "size", "angle", "response", "octave")], 1),
                    d_desc[:n].cpu().numpy().astype(np.float32))
        out = dict(zip(("keypoints", "descriptors"), keypoints(self.d_kps[cur], self.d_desc[cur], last.pop("num_keypoints"))))
        if "num_keypoints_right" in last:
            out.update(zip(("keypoints_right", "descriptors_right"), keypoints(self.d_kps_r, self.d_desc_r, last.pop("num_keypoints_right"))))
        if self.cfg["ba"]:
            last.update(zip(("local_ba_poses", "local_ba_points", "local_ba_outliers"), (a.cpu().numpy() for a in self.d_ba_out)))
        for name, a in last.items():
            a = np.asarray(a)
            out[name] = a if a.dtype == np.float64 else a.astype(np.float32)
        return out

    def bytes_per_frame(self):
        """host<->device bytes of one e2e frame, counted from the arrays the host entry points copy."""
        cfg, pose = self.cfg, self.wl["pose"]
        W, H, NKP = cfg["W"], cfg["H"], cfg["NKP"]
        nimg = 2 if cfg["stereo"] else 1
        h2d = nimg * W * H
        d2h = nimg * NKP * (28 + 32)
        if cfg["stereo"]:
            h2d += 2 * NKP * (4 + 4 + 4 + 32); d2h += NKP * 8
        else:
            nl = len(self.lmsets[0]["xy"])
            h2d += NKP * (4 + 4 + 4 + 4 + 1 + 32) + nl * (8 + 4 + 4 + 4 + 32 + 4)       # frame index + landmark queries
            d2h += nl * 16
            if cfg["ba"]:
                h2d += 2 * NKP * 32; d2h += NKP * 32                                     # brute force: descriptors up, candidate lists down
        npose = len(pose["inv_sigma_sq"])
        h2d += npose * (24 + 8 + 4 + 4) + 96; d2h += npose + 96 + 128
        if cfg["ba"]:
            ba = self.wl["ba"]
            K, Lm, M = len(ba["poses"]), len(ba["points"]), len(ba["obs_kf"])
            h2d += K * 97 + Lm * 24 + M * 24
            d2h += K * 96 + Lm * 24 + M + 512
        return h2d, d2h

    def close(self):
        for h in (self.ext, self.ext_r, self.mt, self.pj, self.st, self.po, getattr(self, "lba", None), getattr(self, "pba", None)):
            if h is not None:
                h.close()


DUMP_BYTES_MAX = 64 << 20


def dump_outputs(cams, path):
    """Writes CameraStream.outputs() of each stream as <path>/stream<k>_<name>.npy, streams in order while the total stays within
    DUMP_BYTES_MAX (a config-4 stream is about 1.5 MB, so every stream of a default run fits)."""
    os.makedirs(path, exist_ok=True)
    total = 0
    for cs in cams:
        arrays = cs.outputs()
        size = sum(a.nbytes for a in arrays.values())
        if total + size > DUMP_BYTES_MAX:
            break
        for name, a in arrays.items():
            np.save(os.path.join(path, "stream%d_%s.npy" % (cs.sid, name)), a)
        total += size


def run_ours(args):
    import torch
    import torch.distributed as dist
    from openvslam_b200 import _lib, feature
    cfg = CONFIGS[args.config]
    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    W, H, NKP = cfg["W"], cfg["H"], cfg["NKP"]
    S = max(1, args.streams if args.streams > 0 else cfg["streams"])
    ring = args.ring if args.ring > 0 else max(12, int(140e6 / (W * H)) // 6 * 6 + 6)      # > 126 MB of frames: larger than L2
    wl = make_workload(cfg, rank, ring)
    wait = args.wait
    if wait == "auto":   # spin while every driving thread can own a core, yield-poll once they cannot
        wait = "spin" if S * world <= max(1, host_cores() - 2) else "yield"
    L = _lib.lib()
    L.ovs_set_wait_mode({"spin": 0, "block": 1, "yield": 2}[wait])

    # ---- device-resident inputs: ring of frames (> L2), shared read-only by the camera streams of this GPU
    def resident(frames):
        h = torch.empty((len(frames), H, W), dtype=torch.uint8).pin_memory()
        for i, f in enumerate(frames):
            h[i].copy_(torch.from_numpy(f))
        d = torch.empty((len(frames), H, W), dtype=torch.uint8, device=dev)
        d.copy_(h)
        return d, h.numpy()
    d_frames, h_frames = resident(wl["frames"])
    d_frames_r, h_frames_r = resident(wl["frames_right"]) if cfg["stereo"] else (None, None)
    torch.cuda.synchronize()
    ext0 = feature.orb_extractor(feature.orb_params(max_num_keypts=NKP), device=local)
    lmsets = make_landmark_sets(cfg, wl, ext0)
    ext0.close()
    spec = args.spec if args.spec > 0 else 4
    spec2 = max(0, args.spec2)
    # CTAs per cluster of the BA's reduced-system solver: 8 minimises the latency of one call, 2 maximises calls per second when
    # several streams share the GPU (ovs_optimizer_set_cluster_width; same results)
    cluster = args.cluster if args.cluster > 0 else (8 if S == 1 else 2)
    cams = [CameraStream(cfg, sid, local, dev, d_frames, h_frames, d_frames_r, h_frames_r, wl, lmsets, ring, spec, cluster, spec2, args.graphs) for sid in range(S)]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_all(name, lo, hi):
        """every camera stream runs frames lo..hi-1 of `name` on its own host thread (the C ABI releases the GIL)"""
        errs = []

        def work(cs):
            try:
                torch.cuda.set_device(local)
                fn = getattr(cs, name)
                for i in range(lo, hi):
                    fn(i)
            except Exception as e:   # noqa: BLE001
                errs.append(e)
        if S == 1:
            work(cams[0])
        else:
            ths = [threading.Thread(target=work, args=(cs,)) for cs in cams]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        if errs:
            raise errs[0]

    event_ms = {}
    fps = args.frames_per_step

    def timed(name, steps, warmup, offset):
        run_all(name, offset, offset + warmup * fps)
        for cs in cams:
            cs.reset()
        barrier()
        l0 = _lib.launch_count()
        # CUDA events bracket the region as well (every stream of the device is idle at both records, so the device
        # timeline between them is the region): reported next to the host clock as a cross-check
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        run_all(name, offset + warmup * fps, offset + (warmup + steps) * fps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        e1.record(); e1.synchronize()
        event_ms[name] = max_over_ranks(e0.elapsed_time(e1) * 1e-3, dev, world) * 1e3
        launches = _lib.launch_count() - l0
        return max_over_ranks(dt, dev, world), launches

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    t_dev, launches = timed("step_device", args.steps, args.warmup, 0)
    dev_state = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in cams[0].st_dev.items()}   # per-kernel times: stream 0
    dev_stage = cams[0].stage_ms["device"].copy()
    if args.dump_outputs and rank == 0:
        dump_outputs(cams, args.dump_outputs)
    t_e2e, _ = timed("step_host", args.steps, args.warmup, 7)
    host_stage = cams[0].stage_ms["host"].copy()
    clocks = sampler.stop() if sampler else None
    fps_d = fps_h = fps

    # ---- per-frame latency of ONE stream alone on the GPU (what a live SLAM session sees): spin waits, the BA iteration
    #      replayed as a CUDA graph.  Reported next to the throughput figures, not part of `value`.
    latency = None
    if not args.no_latency:
        cs = cams[0]
        L.ovs_set_wait_mode(0)
        if cfg["ba"]:
            cs.pba.set_graphs(True); cs.lba.set_graphs(True)
            cs.pba.set_cluster_width(8); cs.lba.set_cluster_width(8)
        nlat = max(5, min(args.steps, 20))
        lat = {}
        for name in ("step_device", "step_host"):
            for i in range(3):
                getattr(cs, name)(100 + i)
            barrier()
            t0 = time.perf_counter()
            for i in range(nlat):
                getattr(cs, name)(103 + i)
            torch.cuda.synchronize()
            lat[name] = max_over_ranks((time.perf_counter() - t0) / nlat, dev, world)
        latency = {"streams": 1, "frames": nlat, "ms_per_frame_device_resident": round(1e3 * lat["step_device"], 4),
                   "ms_per_frame_e2e": round(1e3 * lat["step_host"], 4), "host_wait": "spin", "cuda_graphs": bool(cfg["ba"])}

    value = aggregate_value(args.steps * fps_d * S, t_dev, world)
    e2e = aggregate_value(args.steps * fps_h * S, t_e2e, world)
    h2d, d2h = cams[0].bytes_per_frame()

    out = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        nf = max(dev_state["frames"], 1)
        ext_us = dev_state["ext_us"] / nf
        names = ("upload", "pyramid", "fast_score", "cell_nms_compact", "tree_distribute", "orient_describe", "download", "total_wall")
        stages = {"extract_" + n: round(float(v), 1) for n, v in zip(names, ext_us)}
        stages.update(pose_optimizer_kernel=round(dev_state["pose_us"] / nf, 1))
        traffic = {}
        for fn in ("r2_dram_traffic.json", "r1_dram_traffic.json"):
            try:
                for k, v in json.load(open(os.path.join(ROOT, "profiles", fn))).items():
                    traffic.setdefault(k, v)
            except Exception:
                pass
        ncu_metrics = {}
        try:
            ncu_metrics = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_metrics.json")))
        except Exception:
            pass
        # FAST score kernel: reads the pyramid once and writes the score map once
        lv, w_, h_ = [], W, H
        for l in range(8):
            lv.append((int(round(W / 1.2 ** l)), int(round(H / 1.2 ** l))))
        fast_bytes = 2 * sum(a * b for a, b in lv)
        fast_us = float(ext_us[2])
        fast_gbs = fast_bytes / (fast_us * 1e-6) / 1e9 if fast_us > 0 else 0.0
        rl_fast = {"kernel": "k_fast_score", "bound": "hbm", "achieved": round(fast_gbs, 2), "peak": hbm_peak, "unit": "GB/s",
                   "frac": round(fast_gbs / hbm_peak, 5), "traffic": traffic.get("k_fast_score"), "peak_source": peak_src,
                   "algorithmic_bytes_per_launch": fast_bytes, "avg_launch_us": round(fast_us, 2)}
        out = {
            "metric": METRIC, "value": round(value, 3), "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(1e3 * t_dev / args.steps, 4), "ms_per_step_cuda_events": round(event_ms.get("step_device", 0.0) / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 (extract, Hamming) + f64 (pose optimiser, local BA)", "data": "synthetic (seeded numpy frames and BA graph; no datasets offline)",
            "config": {"workload": cfg["name"], "streams_per_gpu": S, "frames_per_step_per_stream": fps_d, "lm_speculation_width": spec, "lm_second_batch_width": spec2, "lm_cuda_graphs": bool(args.graphs), "ba_solver_cluster_ctas": cluster if cfg["ba"] else None, "host_wait": wait,
                       "host_cores": host_cores(),
                       "step": "%d frame(s) on each of the %d independent camera streams of a GPU (own handles and CUDA streams, one host thread each)"
                               % (fps_d, S),
                       "l2": "frame ring of %d x %.2f MB = %.0f MB > 126 MB L2" % (ring, W * H / 1e6, ring * W * H / 1e6),
                       "value_path": "whole path, inputs resident in HBM (extract_device, brute_force_match_device, frame_index_create_device, "
                                     "local_ba_prepare_device / run / fetch_device); the projection matcher's landmark arrays and the pose "
                                     "optimiser's observations are host-side map data in both legs",
                       "e2e_path": "host-buffer C ABI, all host<->device copies inside the timed region",
                       "timing": "barrier + synchronize on both sides, max over ranks; host clock of the region (every C-ABI call returns with its "
                                 "stream drained) cross-checked by CUDA events recorded while the device is idle (ms_per_step_cuda_events)"},
            "e2e": {"value": round(e2e, 3), "unit": "frames/s", "ms_per_step": round(1e3 * t_e2e / args.steps, 4),
                    "ms_per_step_cuda_events": round(event_ms.get("step_host", 0.0) / args.steps, 4), "frames_per_step_per_stream": fps_h,
                    "h2d_bytes_per_step": int(h2d) * S * fps_h, "d2h_bytes_per_step": int(d2h) * S * fps_h,
                    "stage_ms_per_frame_stream0": {n: round(float(v) / (args.steps * fps_h), 3) for n, v in zip(STAGES, host_stage) if v > 0}},
            "value_stage_ms_per_frame_stream0": {n: round(float(v) / (args.steps * fps_d), 3) for n, v in zip(STAGES, dev_stage) if v > 0},
            "single_stream_latency": latency,
            "gpu_launches": int(launches),
            "stage_us_per_frame": stages,
            "clocks": clocks,
        }
        if cfg["ba"]:
            # Dominant kernel of the step: the cluster Cholesky of the reduced camera system (FP64; DMMA trailing update and panel
            # GEMM).  Algorithmic flops per factorised system: n^3/3 (factorisation) + 2 n^2 (the two triangular solves).
            nred = int(dev_state["reduced_dim"])
            sol_launches = max(int(dev_state["solver_launches"]), 1)
            sol_us = dev_state["solver_us"] / sol_launches
            sol_flops = (nred ** 3 / 3.0 + 2.0 * nred ** 2) * dev_state["solver_trials"] / sol_launches
            sol_tf = sol_flops / (sol_us * 1e-6) / 1e12 if sol_us > 0 else 0.0
            # FP64 tensor peak: MEASURED_PEAKS.json holds no FP64 figure -> measured now, on this GPU (ovs_probe_fp64_peaks)
            dm, df = C.c_double(0), C.c_double(0)
            _lib.check(L.ovs_probe_fp64_peaks(local, C.byref(dm), C.byref(df)))
            fp64_peak = dm.value
            ham_us = dev_state["match_us"] / max(dev_state["match_calls"], 1)
            ham_bytes = (NKP + NKP) * 32 + NKP * 8
            ham_gbs = ham_bytes / (ham_us * 1e-6) / 1e9 if ham_us > 0 else 0.0
            stages.update(match_hamming_kernel=round(ham_us, 1), local_ba_device=round(dev_state["ba_us"] / nf, 1))
            frame_ms = 1e3 * t_dev / (args.steps * fps_d)
            out["roofline"] = {
                "kernel": "k_ba_cholesky_solve", "bound": "tensor", "achieved": round(sol_tf, 4), "peak": round(fp64_peak, 2), "unit": "TFLOP/s",
                "frac": round(sol_tf / fp64_peak, 5) if fp64_peak > 0 else None, "traffic": traffic.get("k_ba_cholesky_solve"),
                "peak_source": "FP64 DMMA (mma.sync.m8n8k4.f64) whole-chip issue rate measured in this run by ovs_probe_fp64_peaks "
                               "(MEASURED_PEAKS.json has no FP64 entry); DFMA pipe measured alongside: %.2f TFLOP/s" % df.value,
                "algorithmic_flops_per_launch": round(sol_flops), "avg_launch_us": round(sol_us, 2),
                "launches_per_frame": round(sol_launches / nf, 2), "share_of_stream_time": round(dev_state["solver_us"] / nf / (1e3 * frame_ms), 4),
                "reduced_dim": nred, "systems_per_launch": round(dev_state["solver_trials"] / sol_launches, 2),
                "lm_trials_per_frame": round(dev_state["ba_trials"] / nf, 2), "lm_iterations_per_frame": round(dev_state["ba_iterations"] / nf, 2),
                "note": "latency bound, not throughput bound: n dependent pivots (fma -> shuffle -> rsqrt -> mul, ~120 clk each "
                        "measured) put a floor of n x 120 clk = %.1f us under every launch" % (nred * 120 / 1.965e3)}
            # Schur complement (k_ba_schur_chunk + k_ba_schur_final), the GEMM north_star asks the tensor-pipe figure for.  Algorithmic
            # flops per co-observation record and damping value: Y_a = Hpl_a (Hll + lambda I)^-1 (6x3x3) + Y_a Hpl_b' (6x3x6) = 162 FMA.
            sch_us = dev_state["schur_us"] / sol_launches
            sch_flops = 2.0 * 162.0 * dev_state["co_observations"] * dev_state["solver_trials"] / sol_launches
            sch_tf = sch_flops / (sch_us * 1e-6) / 1e12 if sch_us > 0 else 0.0
            out["roofline_schur"] = {
                "kernel": "k_ba_schur_chunk+k_ba_schur_final", "bound": "tensor", "achieved": round(sch_tf, 4), "peak": round(fp64_peak, 2), "unit": "TFLOP/s",
                "frac": round(sch_tf / fp64_peak, 5) if fp64_peak > 0 else None, "traffic": traffic.get("k_ba_schur_chunk"),
                "algorithmic_flops_per_launch": round(sch_flops), "co_observations": int(dev_state["co_observations"]), "avg_launch_us": round(sch_us, 2),
                "share_of_stream_time": round(dev_state["schur_us"] / nf / (1e3 * frame_ms), 4),
                "ncu": ncu_metrics.get("k_ba_schur_chunk"),
                "note": "DMMA m8n8k4 issues 6x6 blocks as 8x8 (56 % of the MMA flops are algorithmic) and B200 runs DMMA at the DFMA rate; the kernel "
                        "is bound by the gathers of the Jacobian blocks and the shared-memory fragment traffic (profiles/README.md)"}
            out["roofline_hamming"] = {
                "kernel": "k_hamming_topk+k_topk_merge", "bound": "hbm", "achieved": round(ham_gbs, 3), "peak": hbm_peak, "unit": "GB/s",
                "frac": round(ham_gbs / hbm_peak, 7), "algorithmic_bytes_per_launch": ham_bytes, "traffic": traffic.get("k_hamming_topk"),
                "avg_launch_us": round(ham_us, 2), "ncu": ncu_metrics.get("k_hamming_topk"),
                "operand_stream_gbs_not_hbm": round(NKP * NKP * 64 / (ham_us * 1e-6) / 1e9, 1) if ham_us > 0 else None,
                "popc32_per_s_not_hbm": round(8.0 * NKP * NKP / (ham_us * 1e-6), 0) if ham_us > 0 else None}
            out["roofline_fast_score"] = rl_fast
        else:
            out["roofline"] = rl_fast
        if not args.no_cpu_baseline and world == 1:
            out["cpu_baseline"] = cpu_baseline(cfg, wl, lmsets, threads=1, budget_s=args.cpu_budget)
            if not args.no_cv2:
                out["cpu_baseline"]["opencv_primitives_not_openvslam"] = cv2_baseline(cfg, wl)
    for cs in cams:
        cs.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------ CPU oracle legs
def oracle_landmark_sets(cfg, wl, O, P):
    """the same landmark construction as make_landmark_sets, from the oracle's own extraction (no GPU on this leg)"""
    class _E:
        def extract(self, img):
            kps, desc, _ = O.extract(img, P)
            return kps, desc
    return make_landmark_sets(cfg, wl, _E())


def oracle_step(O, cfg, wl, lmsets, i, prev_desc, P):
    W, H = cfg["W"], cfg["H"]
    pose = wl["pose"]
    sf = np.array([1.2 ** k for k in range(8)], np.float32)
    kps, desc, pyr = O.extract(wl["frames"][i], P)
    if cfg["stereo"]:
        kps_r, desc_r, _ = O.extract(wl["frames_right"][i], P)
        pyr, pyr_r = O.build_pyramid(wl["frames"][i], P), O.build_pyramid(wl["frames_right"][i], P)   # image_pyramid_ of the two extractors
        O.stereo_compute(pyr, pyr_r, sf, kps, desc, kps_r, desc_r, pose["cam"]["focal_x_baseline"], pose["cam"]["focal_x_baseline"] / pose["cam"]["fx"])
    else:
        if cfg["ba"] and prev_desc is not None:
            O.robust_brute_force_match(desc, prev_desc, None, 0.75)
        frm = O.MatchFrame(kps["x"], kps["y"], kps["octave"], kps["angle"], None, desc, O.om_grid(0, W, 0, H))
        s = lmsets[i % wl["nbase"]]
        xy = s["xy"].copy(); xy[:, 0] = (xy[:, 0] + wl["shifts"][i]) % W
        if cfg["ba"]:
            O.projection_match_frame_and_landmarks(frm, sf, xy, None, s["level"], s["desc"], None, None, 5.0)
        else:
            O.projection_match_current_and_last(frm, sf, 8, np.ones(len(xy), np.uint8), xy, None, s["level"], s["angle"], s["desc"], None, 20.0)
    xr = pose["obs_xr"] if cfg["stereo"] else None
    O.pose_optimize(O.camera(**pose["cam"]), not cfg["stereo"], pose["pts_w"], pose["obs_xy"], xr, pose["inv_sigma_sq"], pose["poses"][0])
    if cfg["ba"]:
        ba = wl["ba"]
        O.local_ba(O.camera(**ba["cam"]), True, ba["poses"], ba["fixed"], ba["points"], ba["obs_kf"], ba["obs_lm"], ba["obs_xy"], None, ba["inv_sigma_sq"])
    return desc


def cpu_run(cfg, wl, lmsets, threads, steps_per_thread):
    """`threads` independent streams, each running `steps_per_thread` frames of the oracle (+ one priming frame)."""
    from oracle import oracle as O
    O.build()
    O.lib()
    P = O.params(cfg["NKP"])
    if lmsets is None:
        lmsets = oracle_landmark_sets(cfg, wl, O, P)
    nfr = len(wl["frames"])

    def worker(tid):
        prev = None
        for s in range(steps_per_thread + 1):  # first frame primes prev_desc (its untimed share is small and identical per thread)
            prev = oracle_step(O, cfg, wl, lmsets, (tid + s) % nfr, prev, P)

    ths = [threading.Thread(target=worker, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return threads * (steps_per_thread + 1) / dt, dt, lmsets


def cpu_baseline(cfg, wl, lmsets, threads=1, budget_s=20.0):
    fps, dt, lmsets = cpu_run(cfg, wl, lmsets, threads, 1)
    steps = 1
    if dt < budget_s / 3:
        steps = max(1, int(budget_s / (dt / 2)) - 1)
        fps, dt, _ = cpu_run(cfg, wl, lmsets, threads, steps)
    return {"value": round(fps, 4), "unit": "frames/s", "cores": threads, "kind": "port",
            "sample": "%d frame(s) of the same workload through oracle/ (restated CPU path, gcc -O3 -march=x86-64-v3, single thread), %.1f s"
                      % ((steps + 1) * threads, dt),
            "host_cores_available": host_cores()}


def cv2_baseline(cfg, wl, budget_s=5.0):
    """The OpenCV primitives the reference calls (NOT OpenVSLAM: no cells, tree, orientation or BA), one thread: pyramid resize, FAST
    per level, 7x7 Gaussian blur per level, and a 4000 x 4000 brute-force Hamming match -- a lower bound on the reference's
    front-end cost with a vectorised, production-quality CPU implementation."""
    try:
        import cv2
    except Exception as e:   # noqa: BLE001
        return {"unavailable": str(e)}
    cv2.setNumThreads(1)
    fast = cv2.FastFeatureDetector_create(threshold=20, nonmaxSuppression=True)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    rng = np.random.default_rng(0)
    d1 = rng.integers(0, 256, (cfg["NKP"], 32), dtype=np.uint8); d2 = rng.integers(0, 256, (cfg["NKP"], 32), dtype=np.uint8)
    n, t_front, t_match = 0, 0.0, 0.0
    t_end = time.perf_counter() + budget_s
    while time.perf_counter() < t_end or n < 2:
        img = wl["frames"][n % len(wl["frames"])]
        t0 = time.perf_counter()
        lvl = img
        for l in range(8):
            if l:
                lvl = cv2.resize(lvl, (int(round(cfg["W"] / 1.2 ** l)), int(round(cfg["H"] / 1.2 ** l))), interpolation=cv2.INTER_LINEAR)
            fast.detect(lvl, None)
            cv2.GaussianBlur(lvl, (7, 7), 2, 2, borderType=cv2.BORDER_REFLECT_101)
        t1 = time.perf_counter()
        bf.knnMatch(d1, d2, k=2)
        t2 = time.perf_counter()
        t_front += t1 - t0; t_match += t2 - t1; n += 1
    return {"frames": n, "threads": 1, "ms_per_frame_pyramid_fast_blur": round(1e3 * t_front / n, 3), "ms_per_frame_bfmatcher_knn2": round(1e3 * t_match / n, 3),
            "label": "OpenCV %s primitives only, not the reference's pipeline" % cv2.__version__}


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return None
    cfg = CONFIGS[args.config]
    wl = make_workload(cfg, 0, 6)
    threads = min(host_cores(), args.ref_threads) if args.ref_threads > 0 else host_cores()
    total = args.steps + args.warmup
    per_thread = max(1, (total + threads - 1) // threads)
    fps, dt, _ = cpu_run(cfg, wl, None, threads, per_thread)
    return {
        "impl": "reference", "metric": METRIC, "value": round(fps, 4), "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 / fps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8 + f64",
        "data": "synthetic", "config": {"workload": cfg["name"]},
        "cpu_baseline": {"value": round(fps, 4), "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": "%d independent streams x %d frames through oracle/ (restated CPU path, gcc -O3 -march=x86-64-v3; the reference itself "
                                   "cannot be built: no source in /root/reference), %.1f s" % (threads, per_thread + 1, dt)},
        "e2e": {"value": round(fps, 4), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS), help="BASELINE.json configs[n-1]; 4 = the metric's configuration")
    ap.add_argument("--ring", type=int, default=0, help="frames in the device ring (0: just above 126 MB, the L2 size)")
    ap.add_argument("--streams", type=int, default=0, help="independent camera streams per GPU (0: the config's default, 8; config 5: 1)")
    ap.add_argument("--frames-per-step", type=int, default=8,
                    help="frames per stream per step (default 8: the default 20 steps then time 160 frames on each stream)")
    ap.add_argument("--spec", type=int, default=0, help="local BA speculation width 1..4 (0 = default 4)")
    ap.add_argument("--spec2", type=int, default=0, help="local BA: width of a statically enqueued second trial batch (0 = none)")
    ap.add_argument("--graphs", action="store_true", help="local BA: replay the Levenberg iteration as a CUDA graph in the throughput legs too (default: only in the single-stream latency pass)")
    ap.add_argument("--cluster", type=int, default=0, help="CTAs per cluster of the BA's reduced-system solver (0: 8 for one stream, 2 for several)")
    ap.add_argument("--wait", default="auto", choices=["auto", "spin", "block", "yield"], help="host wait mode (auto: spin while streams x ranks fit the usable cores, else yield-poll)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cv2", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the single-stream latency pass")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--ref-threads", type=int, default=0, help="CPU arm: independent streams (0 = one per usable host core, cgroup quota respected)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the value leg returned for the last frame of each camera stream as DIR/*.npy")
    args = ap.parse_args()
    if args.frames_per_step < 1:
        ap.error("--frames-per-step must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    out = run_reference(args) if args.impl == "reference" else run_ours(args)
    if out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
