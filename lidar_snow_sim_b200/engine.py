"""
SnowfallEngine -- thin host-side owner of one C-ABI engine (one GPU).  PyTorch is used only as the device container
(tensors, streams); all arithmetic happens in liblss_b200.so.

One process per GPU: create one engine per rank; clouds are independent, so a batch shards across ranks with no
data-path collective (see lidar_snow_sim_b200/distributed.py for the gather of the augmented batch).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .calib.hdl64e_s3 import sensor_arrays

DEFAULT_MAX_DIVERGENCE_RAD = 3e-3          # callers pass beam_divergence = degrees(3e-3) (precompute.py:104)


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        return ctypes.c_void_p(t.data_ptr())
    if isinstance(t, np.ndarray):
        return ctypes.c_void_p(t.ctypes.data)
    raise TypeError(type(t))


class SnowfallEngine:
    def __init__(self, device=0, sensor_table=None, camera=None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError('SnowfallEngine needs a CUDA device (no CPU fallback)')
        self.device = torch.device('cuda', device)
        h = ctypes.c_void_p()
        _lib.check(self.lib.lss_create(device, ctypes.byref(h)))
        self.h = h
        fd, fs, mi, mx = sensor_arrays(sensor_table)
        self._sensor = [np.ascontiguousarray(a, dtype=np.float64) for a in (fd, fs, mi, mx)]
        _lib.check(self.lib.lss_set_sensor(self.h, len(fd), *[_ptr(a) for a in self._sensor]), self.h)
        if camera is None:
            from .calib.dense_camera import STF_HDL64_CAMERA as camera
        self.set_camera(camera)
        self._tables = {}
        self._ws = None

    # ------------------------------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, 'h', None):
            self.lib.lss_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def set_camera(self, camera):
        P2 = np.ascontiguousarray(camera['P2'], dtype=np.float32).reshape(3, 4)
        R0 = np.ascontiguousarray(camera['R0'], dtype=np.float32).reshape(3, 3)
        V2C = np.ascontiguousarray(camera['V2C'], dtype=np.float32).reshape(3, 4)
        h, w = camera.get('img_shape', (1024, 1920))
        _lib.check(self.lib.lss_set_camera(self.h, _ptr(P2), _ptr(R0), _ptr(V2C), int(h), int(w)), self.h)

    # ------------------------------------------------------------------------------------------------------------------
    def upload_tables(self, tables, max_beam_divergence_rad=DEFAULT_MAX_DIVERGENCE_RAD, n_buckets=2048):
        """tables: sequence of float64 (Np_k, 3) arrays (x, y, r); plane index k <-> file '<prefix>_<k+1>.npy'."""
        off = np.zeros(len(tables) + 1, dtype=np.int64)
        for k, t in enumerate(tables):
            t = np.asarray(t)
            if t.ndim != 2 or t.shape[1] != 3:
                raise ValueError('particle table must be (N, 3)')
            off[k + 1] = off[k] + t.shape[0]
        xyr = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.float64) for t in tables], axis=0))
        tid = ctypes.c_int(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lss_upload_particles(self.h, len(tables), _ptr(xyr), _ptr(off),
                                                     float(max_beam_divergence_rad), int(n_buckets), self._stream(),
                                                     ctypes.byref(tid)), self.h)
        self._tables[tid.value] = dict(n_planes=len(tables), max_div=float(max_beam_divergence_rad))
        return tid.value

    def upload_tables_device(self, xyr, plane_offsets, max_beam_divergence_rad=DEFAULT_MAX_DIVERGENCE_RAD,
                             n_buckets=2048):
        """xyr: CUDA float64 tensor (sum Np, 3); plane_offsets: int64 host array (n_planes + 1)."""
        off = np.ascontiguousarray(plane_offsets, dtype=np.int64)
        assert xyr.is_cuda and xyr.dtype == torch.float64 and xyr.is_contiguous()
        tid = ctypes.c_int(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lss_upload_particles_device(self.h, len(off) - 1, _ptr(xyr), _ptr(off),
                                                            float(max_beam_divergence_rad), int(n_buckets),
                                                            self._stream(), ctypes.byref(tid)), self.h)
        self._tables[tid.value] = dict(n_planes=len(off) - 1, max_div=float(max_beam_divergence_rad))
        return tid.value

    def sample_tables_device(self, mode, snowfall_rate, terminal_velocity, seed=1000, R_0=80.0, n_planes=64,
                             upload=True, max_beam_divergence_rad=DEFAULT_MAX_DIVERGENCE_RAD, n_buckets=2048,
                             return_candidates=False):
        """
        Draw the n_planes snowflake tables of one (snowfall_rate, terminal_velocity) configuration ON THE DEVICE
        (greedy dart throwing, tools/snowfall/sampling.py:90-194, counter-based random stream) and, with `upload`,
        build the candidate index from them without a host round trip.  Returns the table id, or with upload=False
        (xyr (sum N, 3) CUDA float64 tensor, plane_offsets int64 array[, candidates]).
        """
        from .snowfall.sampling import compute_occupancy, snowfall_rate_to_rainfall_rate, _expected_capacity, _DIST
        if mode not in _DIST:
            raise NotImplementedError('Distribution model unknown.')
        occ = compute_occupancy(float(snowfall_rate), float(terminal_velocity))
        rr = float(snowfall_rate_to_rainfall_rate(float(snowfall_rate), float(terminal_velocity)))
        cap = _expected_capacity(occ, rr, R_0, mode)
        with torch.cuda.device(self.device):
            while True:
                M = cap
                need = self.lib.lss_sample_particles_workspace_bytes(n_planes, M)
                ws = torch.empty(int(need) + 256, dtype=torch.uint8, device=self.device)
                out = torch.empty((n_planes, cap, 3), dtype=torch.float64, device=self.device)
                counts = torch.empty((n_planes,), dtype=torch.int32, device=self.device)
                cand = torch.empty((n_planes, M, 3), dtype=torch.float64, device=self.device) if return_candidates else None
                st = self.lib.lss_sample_particles(self.h, n_planes, occ, rr, float(R_0), _DIST[mode], int(seed), M,
                                                   _ptr(out), cap, _ptr(counts), _ptr(cand), _ptr(ws), int(ws.numel()),
                                                   self._stream())
                if st == _lib.LSS_ERR_WORKSPACE:
                    cap *= 2
                    continue
                _lib.check(st, self.h)
                break
            cnt = counts.cpu().numpy().astype(np.int64)
            off = np.concatenate([[0], np.cumsum(cnt)])
            xyr = torch.cat([out[p, :cnt[p]] for p in range(n_planes)], dim=0).contiguous()
        if not upload:
            return (xyr, off, cand) if return_candidates else (xyr, off)
        return self.upload_tables_device(xyr, off, max_beam_divergence_rad, n_buckets)

    def free_tables(self, table_id):
        _lib.check(self.lib.lss_free_particles(self.h, int(table_id)), self.h)
        self._tables.pop(table_id, None)

    def table_info(self, table_id):
        a, b, c = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        _lib.check(self.lib.lss_table_info(self.h, int(table_id), ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)),
                   self.h)
        return dict(n_particles=a.value, n_entries=b.value, bytes=c.value)

    # ------------------------------------------------------------------------------------------------------------------
    def _workspace(self, n_total, n_clouds):
        need = self.lib.lss_snowfall_workspace_bytes(int(n_total), int(n_clouds))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(int(need * 1.25) + 256, dtype=torch.uint8, device=self.device)
        return self._ws, need

    def snowfall_batch(self, table_id, points, cloud_offsets, order, beam_divergence_deg, theta=None,
                       thresh_poly=None, plane=None, ymins=None, noise_floor=0.7, threshold_filter=True, camera_fov=False,
                       device_prepass=False, assume_sorted=False, want_full=False, want_perm=False, want_nocc=False,
                       out=None, workspace=None):
        """
        Batched augment() on device-resident clouds (enqueued on torch's current stream, no synchronisation).

        points: CUDA float32 (N, 5); cloud_offsets: int64 host array (B + 1); order: int32 host (B, 64).
        plane (B,4) / ymins (B,50): optional host arrays replayed by the device pre-pass (lss_noise_threshold_poly).
        Returns dict(points=(N,5) slot-compacted rows, counts=(B,), stats=(B,4) [, full, perm, nocc]).
        Call `check()` (synchronises) to surface asynchronous device errors.
        """
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous()
        off = np.ascontiguousarray(cloud_offsets, dtype=np.int64)
        B = off.shape[0] - 1
        N = int(off[-1])
        assert points.shape[0] == N and points.shape[1] == 5
        order = np.ascontiguousarray(order, dtype=np.int32).reshape(B, 64)
        flags = 0
        if threshold_filter:
            flags |= _lib.FLAG_THRESHOLD_FILTER
        if camera_fov:
            flags |= _lib.FLAG_CAMERA_FOV
        if device_prepass:
            flags |= _lib.FLAG_DEVICE_PREPASS
        if assume_sorted:
            flags |= _lib.FLAG_ASSUME_SORTED
        want_full = want_full or want_perm or want_nocc      # the debug views are produced together
        tp = None
        if thresh_poly is not None:
            tp = np.ascontiguousarray(thresh_poly, dtype=np.float64).reshape(B, 3)
        if theta is not None:
            assert theta.is_cuda and theta.dtype == torch.float32 and theta.shape[0] == N
        pl = None if plane is None else np.ascontiguousarray(plane, dtype=np.float64).reshape(B, 4)
        ym = None if ymins is None else np.ascontiguousarray(ymins, dtype=np.int32).reshape(B, 50)
        with torch.cuda.device(self.device):
            if out is None:
                out = {}
            if 'points' not in out:
                out['points'] = torch.empty((N, 5), dtype=torch.float32, device=self.device)
                out['counts'] = torch.empty((B,), dtype=torch.int32, device=self.device)
                out['stats'] = torch.empty((B, 4), dtype=torch.float64, device=self.device)
            if want_full and 'full' not in out:
                out['full'] = torch.empty((N, 5), dtype=torch.float32, device=self.device)
            if want_perm and 'perm' not in out:
                out['perm'] = torch.empty((N,), dtype=torch.int32, device=self.device)
            if want_nocc and 'nocc' not in out:
                out['nocc'] = torch.empty((N,), dtype=torch.int32, device=self.device)
            if workspace is None:
                ws, need = self._workspace(N, B)
            else:
                ws = workspace
                assert ws.numel() >= self.lib.lss_snowfall_workspace_bytes(N, B)
            st = self.lib.lss_snowfall_batch(
                self.h, int(table_id), _ptr(points), _ptr(off), B, _ptr(order), float(beam_divergence_deg),
                _ptr(theta), _ptr(tp), _ptr(pl), _ptr(ym), float(noise_floor), flags, _ptr(out['points']),
                _ptr(out['counts']),
                _ptr(out['stats']), _ptr(out.get('full')) if want_full else None,
                _ptr(out.get('perm')) if want_perm else None, _ptr(out.get('nocc')) if want_nocc else None,
                _ptr(ws), int(ws.numel()), self._stream())
        _lib.check(st, self.h)
        return out

    def snowfall_batch_host_submit(self, table_id, host_points, cloud_offsets, order, beam_divergence_deg,
                                   host_out=None, n_chunks=4, thresh_poly=None, noise_floor=0.7, threshold_filter=True,
                                   camera_fov=False, device_prepass=False):
        """
        Enqueue a host-to-host batched augment() (`lss_snowfall_batch_host_submit`) and return a ticket for
        `snowfall_batch_host_wait`.  `host_points`: CPU float32 (N, 5) tensor or numpy array (pinned memory gives full
        PCIe speed).  The batch is cut into `n_chunks` groups of whole clouds that flow through the engine's native
        pipeline (H2D copy, pre-pass, beam stage, D2H copy on separate streams).  Up to 3 batches may be in flight; with
        2-3 in flight (a prefetching loader) batch k+1's copy-in, batch k's kernels and batch k-1's copy-out overlap.
        The input and `host_out` buffers must not be touched until the ticket has been waited for.
        """
        off = np.ascontiguousarray(cloud_offsets, dtype=np.int64)
        B = off.shape[0] - 1
        N = int(off[-1])
        if isinstance(host_points, np.ndarray):
            host_points = torch.from_numpy(np.ascontiguousarray(host_points, dtype=np.float32))
        assert not host_points.is_cuda and host_points.dtype == torch.float32 and host_points.shape == (N, 5)
        assert host_points.is_contiguous()
        order = np.ascontiguousarray(order, dtype=np.int32).reshape(B, 64)
        tp = None
        if thresh_poly is not None:
            tp = np.ascontiguousarray(thresh_poly, dtype=np.float64).reshape(B, 3)
        flags = 0
        if threshold_filter:
            flags |= _lib.FLAG_THRESHOLD_FILTER
        if camera_fov:
            flags |= _lib.FLAG_CAMERA_FOV
        if device_prepass:
            flags |= _lib.FLAG_DEVICE_PREPASS
        if host_out is None:
            host_out = {}
        if 'points' not in host_out:
            host_out['points'] = torch.empty((N, 5), dtype=torch.float32).pin_memory()
            host_out['counts'] = torch.empty((B,), dtype=torch.int32).pin_memory()
            host_out['stats'] = torch.empty((B, 4), dtype=torch.float64).pin_memory()
        assert host_out['points'].shape == (N, 5) and host_out['counts'].shape == (B,)
        ticket = ctypes.c_int(-1)
        st = self.lib.lss_snowfall_batch_host_submit(
            self.h, int(table_id), _ptr(host_points), _ptr(off), B, _ptr(order), float(beam_divergence_deg), _ptr(tp),
            float(noise_floor), flags, int(n_chunks), _ptr(host_out['points']), _ptr(host_out['counts']),
            _ptr(host_out['stats']), ctypes.byref(ticket))
        _lib.check(st, self.h)
        # the ticket keeps the buffers of the in-flight batch alive
        return dict(id=int(ticket.value), out=host_out, keep=(host_points, off, order, tp))

    def snowfall_batch_host_wait(self, ticket):
        """Block until the batch is in its host buffers; raises what the reference would have raised for it.
        Returns dict(points, counts, stats): pinned CPU tensors, slot-compacted layout of snowfall_batch."""
        _lib.check(self.lib.lss_snowfall_batch_host_wait(self.h, int(ticket['id'])), self.h)
        return ticket['out']

    def snowfall_batch_host(self, table_id, host_points, cloud_offsets, order, beam_divergence_deg, **kw):
        """Synchronous host-to-host batched augment(): submit + wait (see snowfall_batch_host_submit)."""
        return self.snowfall_batch_host_wait(
            self.snowfall_batch_host_submit(table_id, host_points, cloud_offsets, order, beam_divergence_deg, **kw))

    def host_pipeline_trace(self, max_chunks=64):
        """Device timeline (ms since call start) of the last snowfall_batch_host call: rows (n_chunks, 4) =
        rows landed, polynomial ready, beam stage done, results on host."""
        buf = np.zeros((max_chunks, 4), dtype=np.float32)
        n = self.lib.lss_host_pipe_trace(self.h, _ptr(buf), max_chunks)
        return buf[:n]

    def noise_threshold_poly(self, points, cloud_offsets, noise_floor=0.7, plane=None, ymins=None, want_fits=False):
        """Device pre-pass only: returns (poly (B,3) float64 tensor in np.polyfit order, plane (B,4) tensor)
        [, fits (B,8) float64, picks (B,50) int32 with want_fits].
        plane: optional host array (B,4) = (w0, w1, w2, h) to use instead of the RANSAC estimate;
        ymins: optional host int array (B,50), the reference host's np.argpartition picks (augmentation.py:236)."""
        off = np.ascontiguousarray(cloud_offsets, dtype=np.int64)
        B = off.shape[0] - 1
        N = int(off[-1])
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous() and points.shape == (N, 5)
        pl = None if plane is None else np.ascontiguousarray(plane, dtype=np.float64).reshape(B, 4)
        ym = None if ymins is None else np.ascontiguousarray(ymins, dtype=np.int32).reshape(B, 50)
        with torch.cuda.device(self.device):
            need = self.lib.lss_prepass_workspace_bytes(N, B)
            ws = torch.empty(int(need) + 256, dtype=torch.uint8, device=self.device)
            poly = torch.empty((B, 3), dtype=torch.float64, device=self.device)
            plane_out = torch.empty((B, 4), dtype=torch.float64, device=self.device)
            fits = torch.empty((B, 8), dtype=torch.float64, device=self.device) if want_fits else None
            picks = torch.empty((B, 50), dtype=torch.int32, device=self.device) if want_fits else None
            st = self.lib.lss_noise_threshold_poly(self.h, _ptr(points), _ptr(off), B, float(noise_floor), _ptr(pl),
                                                   _ptr(ym), _ptr(poly), _ptr(plane_out), _ptr(fits), _ptr(picks),
                                                   _ptr(ws), int(ws.numel()), self._stream())
        _lib.check(st, self.h)
        if want_fits:
            return poly, plane_out, fits, picks
        return poly, plane_out

    def wet_ground_batch(self, points, cloud_offsets, counts=None, water_height=0.001, pavement_depth=0.0012,
                         noise_floor=0.7, power_factor=15, flat_earth=False, delta=0.5, replace=True, plane=None,
                         want_intensity64=False, ymins=None, out=None):
        """
        Batched ground_water_augmentation() on device-resident clouds (current stream, no synchronisation).
        counts: optional CUDA int32 (B,) valid rows per cloud slot (fused snow -> wet path).
        Returns dict(points (N,5) float32 slot-compacted, counts (B,), passthrough (B,), plane (B,4) [, intensity64]).
        """
        off = np.ascontiguousarray(cloud_offsets, dtype=np.int64)
        B = off.shape[0] - 1
        N = int(off[-1])
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous() and points.shape == (N, 5)
        pl = None if plane is None else np.ascontiguousarray(plane, dtype=np.float64).reshape(B, 4)
        ym = None if ymins is None else np.ascontiguousarray(ymins, dtype=np.int32).reshape(B, 50)
        with torch.cuda.device(self.device):
            if out is None:
                out = {}
            if 'points' not in out:                            # (pass the returned dict back in as `out` to reuse the buffers)
                out.update(points=torch.empty((N, 5), dtype=torch.float32, device=self.device),
                           counts=torch.empty((B,), dtype=torch.int32, device=self.device),
                           passthrough=torch.empty((B,), dtype=torch.int32, device=self.device),
                           plane=torch.empty((B, 4), dtype=torch.float64, device=self.device))
            if want_intensity64 and 'intensity64' not in out:
                out['intensity64'] = torch.empty((N,), dtype=torch.float64, device=self.device)
            need = self.lib.lss_wet_ground_workspace_bytes(N, B)
            if getattr(self, '_ws_wet', None) is None or self._ws_wet.numel() < need:
                self._ws_wet = torch.empty(int(need * 1.25) + 256, dtype=torch.uint8, device=self.device)
            st = self.lib.lss_wet_ground_batch(
                self.h, _ptr(points), _ptr(off), _ptr(counts), B, float(water_height), float(pavement_depth),
                float(noise_floor), float(power_factor), 1 if flat_earth else 0, float(delta), 1 if replace else 0,
                _ptr(pl), _ptr(ym), _ptr(out['points']), _ptr(out.get('intensity64')) if want_intensity64 else None,
                _ptr(out['counts']),
                _ptr(out['passthrough']), _ptr(out['plane']), _ptr(self._ws_wet), int(self._ws_wet.numel()),
                self._stream())
        _lib.check(st, self.h)
        return out

    def fog_batch(self, points, cloud_offsets, lut, alpha, beta, beta_0, hard=True, soft=True, gain=False, noise=0,
                  noise_variant=1, rng_states=None, ext_noise=None, want_rank=False):
        """
        Batched simulate_fog() (lib/LiDAR_fog_sim/fog_simulation.py:299-316) on device-resident clouds (current stream,
        no synchronisation).  points: CUDA float32 (N, F), F >= 4; lut: CUDA float64 (2001, 2) integral look-up table;
        rng_states: host uint64 (B, 4) PCG64 states (variants 1-3) or ext_noise: CUDA float64 (N,) values by rank.
        Returns dict(points float64 (N, F), fog_mask uint8 (N,), info float64 (B, 3) [, rank int32 (N,)]).
        """
        off = np.ascontiguousarray(cloud_offsets, dtype=np.int64)
        B = off.shape[0] - 1
        N = int(off[-1])
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous() and points.shape[0] == N
        F = int(points.shape[1])
        if lut is not None:
            assert lut.is_cuda and lut.dtype == torch.float64 and lut.is_contiguous() and tuple(lut.shape) == (2001, 2)
        rs = None if rng_states is None else np.ascontiguousarray(rng_states, dtype=np.uint64).reshape(B, 4)
        if ext_noise is not None:
            assert ext_noise.is_cuda and ext_noise.dtype == torch.float64 and ext_noise.numel() >= N
        flags = (_lib.FOG_HARD if hard else 0) | (_lib.FOG_SOFT if soft else 0) | (_lib.FOG_GAIN if gain else 0)
        with torch.cuda.device(self.device):
            out = dict(points=torch.empty((N, F), dtype=torch.float64, device=self.device),
                       fog_mask=torch.empty((N,), dtype=torch.uint8, device=self.device),
                       info=torch.empty((B, 3), dtype=torch.float64, device=self.device))
            if want_rank:
                out['rank'] = torch.empty((N,), dtype=torch.int32, device=self.device)
            need = self.lib.lss_fog_workspace_bytes(N, B)
            ws = torch.empty(int(need) + 256, dtype=torch.uint8, device=self.device)
            st = self.lib.lss_fog_batch(self.h, _ptr(points), F, _ptr(off), B, float(alpha), float(beta), float(beta_0),
                                        _ptr(lut), flags, int(noise), int(noise_variant), _ptr(rs), _ptr(ext_noise),
                                        _ptr(out['points']), _ptr(out['fog_mask']), _ptr(out.get('rank')),
                                        _ptr(out['info']), _ptr(ws), int(ws.numel()), self._stream())
        _lib.check(st, self.h)
        return out

    def voxelize_batch(self, points, cloud_offsets, point_cloud_range, voxel_size, max_points_per_voxel, max_voxels,
                       counts=None, mask_xy_range=True):
        """
        Batched point-range mask + voxelisation (DataProcessor.mask_points_and_boxes_outside_range +
        transform_points_to_voxels, lib/OpenPCDet/pcdet/datasets/processor/data_processor.py:78-91,115-143) on
        device-resident clouds (current stream, no synchronisation).  points: CUDA float32 (N, F); counts: optional CUDA
        int32 (B,) valid rows per cloud slot.  Returns dict(voxels (B, max_voxels, max_points, F) float32, coords
        (B, max_voxels, 4) int32 = (cloud, z, y, x), num_points (B, max_voxels) int32, n_voxels (B,) int32).
        """
        off = np.ascontiguousarray(cloud_offsets, dtype=np.int64)
        B = off.shape[0] - 1
        N = int(off[-1])
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous() and points.shape[0] == N
        F = int(points.shape[1])
        rng = np.ascontiguousarray(point_cloud_range, dtype=np.float32).reshape(6)
        vs = np.ascontiguousarray(voxel_size, dtype=np.float32).reshape(3)
        T, MV = int(max_points_per_voxel), int(max_voxels)
        with torch.cuda.device(self.device):
            out = dict(voxels=torch.empty((B, MV, T, F), dtype=torch.float32, device=self.device),
                       coords=torch.empty((B, MV, 4), dtype=torch.int32, device=self.device),
                       num_points=torch.empty((B, MV), dtype=torch.int32, device=self.device),
                       n_voxels=torch.empty((B,), dtype=torch.int32, device=self.device))
            need = self.lib.lss_voxelize_workspace_bytes(N, B, T, MV)
            if getattr(self, '_ws_vox', None) is None or self._ws_vox.numel() < need:
                self._ws_vox = torch.empty(int(need * 1.25) + 256, dtype=torch.uint8, device=self.device)
            st = self.lib.lss_voxelize_batch(self.h, _ptr(points), F, _ptr(off), _ptr(counts), B, _ptr(rng), _ptr(vs), T, MV,
                                             1 if mask_xy_range else 0, _ptr(out['voxels']), _ptr(out['coords']),
                                             _ptr(out['num_points']), _ptr(out['n_voxels']), _ptr(self._ws_vox),
                                             int(self._ws_vox.numel()), self._stream())
        _lib.check(st, self.h)
        return out

    def dror_batch(self, points, cloud_offsets, counts=None, alpha=0.16, beta=3.0, k_min=3, sr_min=0.04, crop_xy=None,
                   compact=True, out=None):
        """
        Dynamic radius outlier removal (dynamic_radius_outlier_filter, lib/cadc_devkit/other/dror.py:288-334) of every
        cloud of a batch, on the current stream without synchronisation.  points: CUDA float32 (N, F), F >= 3;
        cloud_offsets: host int64 (B + 1); counts: optional CUDA int32 (B,) valid rows per cloud slot (the slot-compacted
        output of snowfall_batch / wet_ground_batch); crop_xy: optional (x0, x1, y0, y1), the `crop` variant
        (get_cube_mask, z ignored).  Returns dict(codes uint8 (N,) 0 snow / 1 kept / 2 outside the crop, points (N, F)
        kept rows slot-compacted (None without `compact`), counts int32 (B,) kept rows, n_snow int32 (B,)).
        """
        off = np.ascontiguousarray(cloud_offsets, dtype=np.int64)
        B = off.shape[0] - 1
        N = int(off[-1])
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous() and points.shape[0] == N
        F = int(points.shape[1])
        if counts is not None:
            assert counts.is_cuda and counts.dtype == torch.int32 and counts.shape[0] == B
        crop = None if crop_xy is None else np.ascontiguousarray(crop_xy, dtype=np.float32).reshape(4)
        with torch.cuda.device(self.device):
            if out is None:
                out = {}
            if 'codes' not in out:                             # (pass the returned dict back in as `out` to reuse the buffers)
                out.update(codes=torch.empty((N,), dtype=torch.uint8, device=self.device),
                           counts=torch.empty((B,), dtype=torch.int32, device=self.device),
                           n_snow=torch.empty((B,), dtype=torch.int32, device=self.device), points=None)
            if compact and out.get('points') is None:
                out['points'] = torch.empty((N, F), dtype=torch.float32, device=self.device)
            need = self.lib.lss_dror_workspace_bytes(N, B)
            if need < 0:
                raise RuntimeError('lss_dror_workspace_bytes failed: no usable CUDA device')
            if getattr(self, '_ws_dror', None) is None or self._ws_dror.numel() < need:
                self._ws_dror = torch.empty(int(need * 1.25) + 256, dtype=torch.uint8, device=self.device)
            st = self.lib.lss_dror_batch(self.h, _ptr(points), F, _ptr(off), _ptr(counts), B, float(alpha), float(beta),
                                         int(k_min), float(sr_min), _ptr(crop), _ptr(out['codes']),
                                         _ptr(out['points']) if compact else None, _ptr(out['counts']),
                                         _ptr(out['n_snow']), _ptr(self._ws_dror), int(self._ws_dror.numel()),
                                         self._stream())
        _lib.check(st, self.h)
        if not compact:
            out['points'] = None
        return out

    def gather_push(self, points, counts, d_cloud_offsets, n_rows, world, rank, peer_points, peer_counts, mc_points=0,
                    mc_counts=0, blocks=0):
        """lss_gather_push on the current stream: write the kept rows of this rank's slot-compacted batch (+ counts) into
        every rank's gathered buffers (SURVEY.md 8e).  peer_points / peer_counts: per rank, a CUDA tensor mapping that
        rank's gathered buffer (world * n_rows, 5) float32 / (world * n_clouds,) int32 into this process (see
        distributed.BatchGather, which owns the symmetric allocations and the side stream)."""
        B = int(d_cloud_offsets.shape[0]) - 1
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous()
        assert d_cloud_offsets.is_cuda and d_cloud_offsets.dtype == torch.int64
        P = ctypes.c_void_p * int(world)
        pp = P(*[t.data_ptr() for t in peer_points])
        pc = P(*[t.data_ptr() for t in peer_counts])
        with torch.cuda.device(self.device):
            st = self.lib.lss_gather_push(self.h, _ptr(points), _ptr(counts), _ptr(d_cloud_offsets), B, int(n_rows), int(world),
                                          int(rank), pp, pc, mc_points or None, mc_counts or None, int(blocks), self._stream())
        _lib.check(st, self.h)

    def check(self):
        """Synchronise the current stream and raise the exception type the reference would have raised."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lss_check_async(self.h, self._stream()), self.h)

    def launch_count(self):
        return int(self.lib.lss_launch_count(self.h))

    def set_profiling(self, enable=True):
        _lib.check(self.lib.lss_set_profiling(self.h, 1 if enable else 0), self.h)

    def kernel_times(self, reset=True):
        """{kernel name: (total ms, launches)} measured with CUDA events on the launching stream (synchronises)."""
        torch.cuda.synchronize(self.device)
        n = 10
        ms = np.zeros(n, dtype=np.float64)
        calls = np.zeros(n, dtype=np.int64)
        _lib.check(self.lib.lss_kernel_times(self.h, 1 if reset else 0, _ptr(ms), _ptr(calls), n), self.h)
        return {self.lib.lss_kernel_name(k).decode(): (float(ms[k]), int(calls[k])) for k in range(n)}


_default_engines = {}


def default_engine(device=None):
    """Process-wide engine per device, created on first use (used by the reference-signature wrappers)."""
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if device not in _default_engines:
        _default_engines[device] = SnowfallEngine(device)
    return _default_engines[device]
