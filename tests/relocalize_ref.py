"""numpy restatement of vloam_b200_relocalize's search (include/vloam_b200.h): query selection, occupancy, per-yaw base cells,
exhaustive scoring, best and runner-up with the lowest-index tie rule.  Every float64 expression is spelled in the order the device
code evaluates it (no FMA, math.cos / math.sin are the libm routines the library calls), so the grids and cells are bit-equal and
the scores, being integer counts, exactly equal."""
import math

import numpy as np


def rot(q):
    """Eigen's toRotationMatrix of q / |q| (q x,y,z,w)."""
    x, y, z, w = [float(v) for v in q]
    n = math.sqrt(((x * x + y * y) + z * z) + w * w)
    x, y, z, w = x / n, y / n, z / n, w / n
    tx, ty, tz = 2 * x, 2 * y, 2 * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz, tyy, tyz, tzz = tx * x, ty * x, tz * x, ty * y, tz * y, tz * z
    R = np.array([[1 - (tyy + tzz), txy - twz, txz + twy], [txy + twz, 1 - (txx + tzz), tyz - twx], [txz - twy, tyz + twx, 1 - (txx + tyy)]])
    return R, np.array([x, y, z, w])


def select(stack_c, stack_s, q, max_range=60.0, max_points=2048):
    """Query points u = R_c p (float64[m, 3]) from the stacks (float32[n, 4])."""
    p = np.concatenate([np.asarray(stack_c, np.float32)[:, :3], np.asarray(stack_s, np.float32)[:, :3]]).astype(np.float64)
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    p = p[x * x + y * y + z * z <= max_range * max_range]
    n = len(p)
    k = -(-n // max_points) if n else 1
    p = p[::k]
    R, _ = rot(q)
    px, py, pz = p[:, 0], p[:, 1], p[:, 2]
    return np.stack([R[i, 0] * px + R[i, 1] * py + R[i, 2] * pz for i in range(3)], axis=1)


class Space:
    """The discretisation of one call (field names as in relocalize.cu's RlSpace)."""

    def __init__(self, u, t_c, half_xy=20.0, half_z=1.0, half_yaw_deg=180.0, resolution=1.0, yaw_step_deg=0.0, max_range=60.0,
                 exclusion_m=3.0, exclusion_deg=10.0):
        r = self.r = float(resolution)
        self.t_c = np.asarray(t_c, np.float64)
        self.dth = yaw_step_deg * math.pi / 180.0 if yaw_step_deg > 0 else r / max_range
        self.full = half_yaw_deg >= 180.0
        if self.full:
            self.nJ, self.j0 = int(math.ceil(2.0 * math.pi / self.dth - 1e-9)), 0
        else:
            J = int(math.floor(half_yaw_deg * math.pi / 180.0 / self.dth + 1e-9))
            self.nJ, self.j0 = 2 * J + 1, J
        self.N, self.Nz = int(math.floor(half_xy / r)), int(math.floor(half_z / r))
        self.S, self.nZ = 2 * self.N + 1, 2 * self.Nz + 1
        zmax = float(np.abs(u[:, 2]).max()) if len(u) else 0.0
        gx = 2 * (int(math.ceil(max_range / r)) + self.N + 1)
        self.dims = np.array([gx, gx, 2 * (int(math.ceil(zmax / r)) + self.Nz + 1)], np.int64)
        self.o = np.array([self.t_c[a] - r * float(self.dims[a] // 2) for a in range(3)])
        self.excl_m, self.excl_rad = exclusion_m, exclusion_deg * math.pi / 180.0
        self.candidates = self.nJ * self.nZ * self.S * self.S

    def theta(self, j):
        return float(j - self.j0) * self.dth

    def yaw_table(self):
        return np.array([[math.cos(self.theta(j)), math.sin(self.theta(j))] for j in range(self.nJ)])

    def occupancy(self, map_pts):
        """uint8[Gz, Gy, Gx]: 1 where a map point (float32[n, >=3]) falls."""
        occ = np.zeros(self.dims[::-1], np.uint8)
        m = np.asarray(map_pts, np.float32)[:, :3].astype(np.float64)
        c = np.floor((m - self.o) / self.r).astype(np.int64)
        ok = np.all((c >= 0) & (c < self.dims), axis=1)
        occ[c[ok, 2], c[ok, 1], c[ok, 0]] = 1
        return occ

    def cells(self, u):
        """int64[nJ, m, 3] base cells c_j(p)."""
        out = np.empty((self.nJ, len(u), 3), np.int64)
        ux, uy, uz = u[:, 0], u[:, 1], u[:, 2]
        for j, (c, s) in enumerate(self.yaw_table()):
            out[j, :, 0] = np.floor(((c * ux - s * uy) + self.t_c[0] - self.o[0]) / self.r)
            out[j, :, 1] = np.floor(((s * ux + c * uy) + self.t_c[1] - self.o[1]) / self.r)
            out[j, :, 2] = np.floor((uz + self.t_c[2] - self.o[2]) / self.r)
        return out

    def scores(self, occ, cells):
        """Exhaustive int64[nJ, nZ, S, S] scores ((j, iz, iy, ix) order: a C-order flat index is the candidate index)."""
        N, Nz = self.N, self.Nz
        flat = cells.reshape(-1, 3)
        lo = np.maximum(-flat.min(axis=0), 0) if len(flat) else np.zeros(3, np.int64)
        hi = np.maximum(flat.max(axis=0) - (self.dims - 1), 0) if len(flat) else np.zeros(3, np.int64)
        px, py, pz = N + 1 + max(lo[0], hi[0]), N + 1 + max(lo[1], hi[1]), Nz + 1 + max(lo[2], hi[2])
        pad = np.zeros((occ.shape[0] + 2 * pz, occ.shape[1] + 2 * py, occ.shape[2] + 2 * px), np.uint8)
        pad[pz:pz + occ.shape[0], py:py + occ.shape[1], px:px + occ.shape[2]] = occ
        off = np.arange(-N, N + 1)
        out = np.zeros((self.nJ, self.nZ, self.S, self.S), np.int64)
        for j in range(self.nJ):
            c = cells[j]
            yy = (c[:, 1] + py)[:, None, None] + off[None, :, None]
            xx = (c[:, 0] + px)[:, None, None] + off[None, None, :]
            for iz in range(self.nZ):
                zz = (c[:, 2] + (iz - Nz) + pz)[:, None, None]
                out[j, iz] = pad[zz, yy, xx].sum(axis=0, dtype=np.int64)
        return out

    def decode(self, lin):
        S, nZ = self.S, self.nZ
        return lin // (nZ * S * S), (lin // (S * S)) % nZ, (lin // S) % S, lin % S

    def in_zone(self, best):
        """bool[nJ, 1, S, S]: candidates inside the runner-up exclusion zone around candidate index `best`."""
        jb, _, ayb, axb = self.decode(best)
        dj = np.abs(np.arange(self.nJ) - jb)
        if self.full:
            dj = np.minimum(dj, self.nJ - dj)
        yaw = dj.astype(np.float64) * self.dth < self.excl_rad
        a = np.arange(self.S)
        dx = np.abs(a - axb).astype(np.float64) * self.r < self.excl_m
        dy = np.abs(a - ayb).astype(np.float64) * self.r < self.excl_m
        return yaw[:, None, None, None] & dy[None, None, :, None] & dx[None, None, None, :]

    def best_and_runner(self, scores):
        """((index, score), (runner index or -1, runner score or -1))."""
        flat = scores.reshape(-1)
        b = int(np.argmax(flat))
        masked = np.where(np.broadcast_to(self.in_zone(b), scores.shape), -1, scores).reshape(-1)
        rI = int(np.argmax(masked))
        return (b, int(flat[b])), ((rI, int(masked[rI])) if masked[rI] >= 0 else (-1, -1))

    def pose(self, lin, q_c):
        """Candidate index -> (q x,y,z,w, t): qz(theta_j) * q_c (the device's quaternion product), t_c + r (ix, iy, iz)."""
        j, iz, ay, ax = self.decode(lin)
        _, qn = rot(q_c)
        th = self.theta(j)
        a = (0.0, 0.0, math.sin(th / 2.0), math.cos(th / 2.0))
        ax_, ay_, az_, aw = a
        bx, by, bz, bw = [float(v) for v in qn]
        q = np.array([aw * bx + ax_ * bw + ay_ * bz - az_ * by, aw * by + ay_ * bw + az_ * bx - ax_ * bz,
                      aw * bz + az_ * bw + ax_ * by - ay_ * bx, aw * bw - ax_ * bx - ay_ * by - az_ * bz])
        t = np.array([self.t_c[0] + self.r * float(ax - self.N), self.t_c[1] + self.r * float(ay - self.N), self.t_c[2] + self.r * float(iz - self.Nz)])
        return q, t


def search(stack_c, stack_s, map_pts, q_c, t_c, max_range=60.0, max_points=2048, **kw):
    """The whole call: returns (space, u, occ, scores, (best, score), (runner, runner score))."""
    u = select(stack_c, stack_s, q_c, max_range, max_points)
    sp = Space(u, t_c, max_range=max_range, **kw)
    occ = sp.occupancy(map_pts)
    sc = sp.scores(occ, sp.cells(u))
    return (sp, u, occ, sc) + sp.best_and_runner(sc)
