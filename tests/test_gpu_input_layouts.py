"""Point layouts the C ABI accepts besides packed XYZ and KITTI's XYZI: any stride >= 3 floats (PointXYZI as PCL pads it is 8),
host or device memory, any float alignment (the scan-registration kernels read float4s only for stride 4 at a 16-byte aligned
address).  Every layout must give the scan-registration outputs of the stride-4 KITTI layout bit for bit, and the same poses."""
import numpy as np
import pytest

from conftest import assert_bits_equal
from test_gpu_parity import KW, SR_NAMES, check_sr

pytestmark = pytest.mark.gpu

N_SWEEPS = 4


def _padded(scan, stride, seed):
    """scan (n, 4) -> (n, stride) float32 with x, y, z first and NaN / garbage in every other field, the intensity slot included."""
    rng = np.random.RandomState(seed)
    out = (rng.randn(len(scan), stride) * 1e6).astype(np.float32)
    out[:, 3::2] = np.nan
    out[:, :3] = scan[:, :3]
    return np.ascontiguousarray(out)


@pytest.fixture(scope="module")
def sweeps(synth, street):
    traj = synth.trajectory(N_SWEEPS + 1)
    return [street.scan(0, traj[k], 1000 + k) for k in range(N_SWEEPS + 1)]


@pytest.fixture(scope="module")
def reference(pkg, sweeps):
    """Stride 4 from host memory, one sweep at a time: poses and the scan-registration outputs of every sweep."""
    g = pkg.Context(**KW[0])
    poses, sr = [], []
    for s in sweeps[:N_SWEEPS]:
        poses.append(g.process_frame(s).copy())
        sr.append({nm: g.get(nm) for nm in SR_NAMES})
    g.close()
    return np.array(poses), sr


def _check_sweep(g, ref_sr, what):
    for nm in SR_NAMES:
        assert_bits_equal(ref_sr[nm], g.get(nm), "%s: %s" % (what, nm))


@pytest.mark.parametrize("stride", [5, 8])
def test_layout_padded_strides_host_and_device(pkg, sweeps, reference, stride):
    import torch
    ref_poses, ref_sr = reference
    padded = [_padded(s, stride, 40 + k) for k, s in enumerate(sweeps)]
    g = pkg.Context(**KW[0])
    for k in range(N_SWEEPS):
        assert (g.process_frame(padded[k]) == ref_poses[k]).all(), "host stride %d, sweep %d" % (stride, k)
        _check_sweep(g, ref_sr[k], "host stride %d sweep %d" % (stride, k))
    g.close()
    dev = [torch.from_numpy(p).cuda() for p in padded]
    g = pkg.Context(**KW[0])
    pose = np.zeros(14)
    for k in range(N_SWEEPS):
        g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], stride, pose.ctypes.data)
        assert (pose == ref_poses[k]).all(), "device stride %d, sweep %d" % (stride, k)
        _check_sweep(g, ref_sr[k], "device stride %d sweep %d" % (stride, k))
    g.close()


def test_layout_misaligned_device_pointer(pkg, sweeps, reference):
    """Stride 4 at an address one float past a 16-byte boundary, through vloam_b200_scan_registration_device itself and through
    process_frame_device: the kernels fall back from float4 to scalar loads."""
    import torch
    ref_poses, ref_sr = reference
    bufs = []
    for s in sweeps[:N_SWEEPS]:
        buf = torch.full((s.size + 4,), float("nan"), dtype=torch.float32, device="cuda")
        buf[1:1 + s.size] = torch.from_numpy(s.ravel()).cuda()
        assert (buf.data_ptr() + 4) % 16 == 4
        bufs.append(buf)
    torch.cuda.synchronize()
    sr_only = pkg.Context(**KW[0])
    g = pkg.Context(**KW[0])
    pose = np.zeros(14)
    for k, buf in enumerate(bufs):
        n = len(sweeps[k])
        sr_only.begin_frame(); sr_only.scan_registration_device(buf.data_ptr() + 4, n, 4)
        _check_sweep(sr_only, ref_sr[k], "scan_registration_device, misaligned, sweep %d" % k)
        g.process_frame_device(buf.data_ptr() + 4, n, 4, pose.ctypes.data)
        assert (pose == ref_poses[k]).all(), "misaligned device pointer, sweep %d" % k
        _check_sweep(g, ref_sr[k], "process_frame_device, misaligned, sweep %d" % k)
    sr_only.close(); g.close()


@pytest.mark.parametrize("device", [True, False], ids=["device", "host"])
def test_layout_lookahead_at_stride_8(pkg, sweeps, reference, device):
    """prefetch_device / prefetch_ptr, two sweeps ahead as bench.prefetch_ahead registers them, with process_frame_device /
    process_frame_ptr at stride 8.  (No debug read between the sweeps: it would drain the look-ahead work.)"""
    import torch
    ref_poses, ref_sr = reference
    padded = [torch.from_numpy(_padded(s, 8, 60 + k)) for k, s in enumerate(sweeps)]
    bufs = [p.cuda() for p in padded] if device else [p.pin_memory() for p in padded]
    g = pkg.Context(**KW[0])
    prefetch, process = (g.prefetch_device, g.process_frame_device) if device else (g.prefetch_ptr, g.process_frame_ptr)
    pose, registered = np.zeros(14), set()
    for k in range(N_SWEEPS):
        for j in (k + 1, k + 2):
            if j <= N_SWEEPS and j not in registered:
                prefetch(bufs[j].data_ptr(), bufs[j].shape[0], 8)
                registered.add(j)
        process(bufs[k].data_ptr(), bufs[k].shape[0], 8, pose.ctypes.data)
        assert (pose == ref_poses[k]).all(), "look-ahead at stride 8, sweep %d" % k
    _check_sweep(g, ref_sr[N_SWEEPS - 1], "look-ahead stride 8, last sweep")
    g.close()


def test_layout_same_pointer_other_stride_is_not_adopted(pkg, sweeps, reference):
    """A sweep registered ahead as (pointer, n, 8) and then processed as (pointer, n, 4): the look-ahead result belongs to
    the other reading of the buffer and must be dropped -- the frame equals a plain run on the stride-4 reading."""
    import torch
    s1 = _padded(sweeps[1], 8, 70)
    as4 = np.ascontiguousarray(s1.ravel()[:len(s1) * 4].reshape(-1, 4))   # the stride-4 reading of the same n points
    want = pkg.Context(**KW[0])
    want.process_frame(sweeps[0])
    want_pose = want.process_frame(as4)
    want_sr = {nm: want.get(nm) for nm in SR_NAMES}
    want.close()
    buf = torch.from_numpy(s1).cuda()
    g = pkg.Context(**KW[0])
    g.process_frame(sweeps[0])
    g.prefetch_device(buf.data_ptr(), len(s1), 8)
    pose = np.zeros(14)
    g.process_frame_device(buf.data_ptr(), len(s1), 4, pose.ctypes.data)
    assert (pose == want_pose).all(), "the stride-8 look-ahead was adopted for a stride-4 call"
    _check_sweep(g, want_sr, "same pointer, other stride")
    # (the stride-4 reading holds every other point of the sweep and a NaN row in between: adopting would be visible)
    assert len(want_sr["sr.laserCloud"]) < len(reference[1][1]["sr.laserCloud"])
    g.close()


@pytest.mark.parametrize("n", [0, 1])
def test_layout_device_call_tiny_clouds(pkg, op, n):
    """n = 0 and n = 1 through vloam_b200_scan_registration_device (stride 4 and 8) against the oracle."""
    import torch
    pts = np.array([[5.0, 0.5, 0.1, 7.0]], np.float32)[:n]
    o = op.Oracle(**KW[0])
    o.scan_registration(pts[:, :3])
    g = pkg.Context(**KW[0])
    for stride in (4, 8):
        buf = torch.zeros(max(n, 1) * stride, dtype=torch.float32, device="cuda")
        if n:
            buf[:3] = torch.from_numpy(pts[0, :3]).cuda()
        g.begin_frame(); g.scan_registration_device(buf.data_ptr(), n, stride)
        check_sr(o, g)
    g.close()
