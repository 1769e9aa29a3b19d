"""On-disk formats the reference node writes (SURVEY.md §8(f) rank 4), so that the engine can be driven from a saved run:

  poses_kitti.txt   one line per keyframe: the 3x4 row-major [R|t]           fast_lio_sam_qn/src/fast_lio_sam_qn.cpp:344-360
  poses_tum.txt     timestamp tx ty tz qx qy qz qw                           fast_lio_sam_qn.cpp:361-376
  pcd/%06d.pcd      the keyframe cloud in the LiDAR frame (x y z intensity)  fast_lio_sam_qn.cpp:349-352 (pcl::io::savePCDFileASCII)
  result.bag        rosbag 2.0: /keyframe_pcd (PointCloud2) + /keyframe_pose (PoseStamped) per keyframe   fast_lio_sam_qn.cpp:377-394
  <seq>_map.pcd     the corrected global map (x y z intensity; Keyframes.build_map)                     fast_lio_sam_qn.cpp:398-411

Host-side I/O only; nothing here is on the hot path.
"""
import os

import numpy as np


def save_poses_kitti(path, poses):
    poses = np.asarray(poses, np.float64).reshape(-1, 4, 4)
    with open(path, "w") as f:
        for T in poses:
            f.write(" ".join("%.17g" % v for v in T[:3, :].reshape(-1)) + "\n")


def load_poses_kitti(path):
    rows = np.loadtxt(path, dtype=np.float64).reshape(-1, 12)
    out = np.tile(np.eye(4), (len(rows), 1, 1))
    out[:, :3, :] = rows.reshape(-1, 3, 4)
    return out


def _quat_to_rot(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _rot_to_quat(R):
    t = np.trace(R)
    if t > 0:
        s = np.sqrt(t + 1.0) * 2
        w, x, y, z = 0.25 * s, (R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s
    else:
        i = int(np.argmax(np.diag(R)))
        j, k = (i + 1) % 3, (i + 2) % 3
        s = np.sqrt(1.0 + R[i, i] - R[j, j] - R[k, k]) * 2
        q = [0.0, 0.0, 0.0]
        q[i] = 0.25 * s
        q[j] = (R[j, i] + R[i, j]) / s
        q[k] = (R[k, i] + R[i, k]) / s
        w = (R[k, j] - R[j, k]) / s
        x, y, z = q
    return np.array([x, y, z, w])


def save_poses_tum(path, stamps, poses):
    poses = np.asarray(poses, np.float64).reshape(-1, 4, 4)
    with open(path, "w") as f:
        for t, T in zip(stamps, poses):
            q = _rot_to_quat(T[:3, :3])
            f.write("%.9f %.17g %.17g %.17g %.17g %.17g %.17g %.17g\n" % (t, T[0, 3], T[1, 3], T[2, 3], q[0], q[1], q[2], q[3]))


def load_poses_tum(path):
    rows = np.loadtxt(path, dtype=np.float64).reshape(-1, 8)
    poses = np.tile(np.eye(4), (len(rows), 1, 1))
    for T, r in zip(poses, rows):
        T[:3, :3] = _quat_to_rot(r[4:8] / np.linalg.norm(r[4:8]))
        T[:3, 3] = r[1:4]
    return rows[:, 0].copy(), poses


def save_pcd(path, pts, binary=False):
    """pts (n, 4): x y z intensity.  ASCII like pcl::io::savePCDFileASCII, or binary."""
    pts = np.ascontiguousarray(pts, np.float32)
    n = len(pts)
    hdr = ("# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z intensity\nSIZE 4 4 4 4\nTYPE F F F F\n"
           "COUNT 1 1 1 1\nWIDTH %d\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS %d\nDATA %s\n" % (n, n, "binary" if binary else "ascii"))
    with open(path, "wb") as f:
        f.write(hdr.encode())
        if binary:
            f.write(pts[:, :4].tobytes())
        else:
            for p in pts:
                f.write(("%.9g %.9g %.9g %.9g\n" % (p[0], p[1], p[2], p[3])).encode())


def load_pcd(path):
    """Reads x y z [intensity] float32 PCD files (ascii or binary, the two forms PCL writes for PointXYZI)."""
    with open(path, "rb") as f:
        fields, sizes, types, counts, npts, data = [], [], [], [], 0, None
        while True:
            line = f.readline().decode("ascii", "replace").strip()
            if not line or line.startswith("#"):
                if not line:
                    break
                continue
            key, _, rest = line.partition(" ")
            if key == "FIELDS":
                fields = rest.split()
            elif key == "SIZE":
                sizes = [int(v) for v in rest.split()]
            elif key == "TYPE":
                types = rest.split()
            elif key == "COUNT":
                counts = [int(v) for v in rest.split()]
            elif key == "POINTS":
                npts = int(rest)
            elif key == "DATA":
                data = rest
                break
        counts = counts or [1] * len(fields)
        if data == "ascii":
            arr = np.loadtxt(f, dtype=np.float64).reshape(npts, -1)
        elif data == "binary":
            rec = sum(s * c for s, c in zip(sizes, counts))
            raw = np.frombuffer(f.read(rec * npts), dtype=np.uint8).reshape(npts, rec)
            cols, off = [], 0
            for s, t, c in zip(sizes, types, counts):
                dt = {("F", 4): np.float32, ("F", 8): np.float64, ("U", 4): np.uint32, ("I", 4): np.int32, ("U", 1): np.uint8,
                      ("U", 2): np.uint16, ("I", 2): np.int16, ("I", 1): np.int8}[(t, s)]
                cols.append(raw[:, off:off + s * c].copy().view(dt).reshape(npts, c).astype(np.float64))
                off += s * c
            arr = np.concatenate(cols, 1)
        else:
            raise ValueError("unsupported PCD DATA section: %r" % data)
    out = np.zeros((npts, 4), np.float32)
    for name, col in (("x", 0), ("y", 1), ("z", 2), ("intensity", 3)):
        if name in fields:
            out[:, col] = arr[:, fields.index(name)]
    return out


def save_run(directory, clouds, poses, stamps, binary=False, map_xyzi=None, seq_name=""):
    """The reference's save layout: <dir>/pcd/%06d.pcd, poses_kitti.txt, poses_tum.txt (fast_lio_sam_qn.cpp:327-413), and
    with map_xyzi (e.g. Keyframes.build_map's records) <dir>/<seq_name>_map.pcd in ASCII, as save_map_pcd writes it (:410)."""
    os.makedirs(os.path.join(directory, "pcd"), exist_ok=True)
    for i, c in enumerate(clouds):
        save_pcd(os.path.join(directory, "pcd", "%06d.pcd" % i), c, binary=binary)
    save_poses_kitti(os.path.join(directory, "poses_kitti.txt"), poses)
    save_poses_tum(os.path.join(directory, "poses_tum.txt"), stamps, poses)
    if map_xyzi is not None:
        save_pcd(os.path.join(directory, "%s_map.pcd" % seq_name), map_xyzi)


def load_run(directory):
    """-> dict(clouds, poses, stamps): feed it to Context.keyframes().add(...) to replay a saved reference run."""
    stamps, poses = load_poses_tum(os.path.join(directory, "poses_tum.txt"))
    kitti = os.path.join(directory, "poses_kitti.txt")
    if os.path.exists(kitti):
        poses = load_poses_kitti(kitti)  # full-precision rotation
    clouds = []
    i = 0
    while os.path.exists(os.path.join(directory, "pcd", "%06d.pcd" % i)):
        clouds.append(load_pcd(os.path.join(directory, "pcd", "%06d.pcd" % i)))
        i += 1
    return dict(clouds=clouds, poses=poses, stamps=stamps)


# ----------------------------------------------------------------------------------------------------------------------
# result.bag (fast_lio_sam_qn.cpp:377-394): rosbag format 2.0 with the two topics the reference writes,
#   /keyframe_pcd   sensor_msgs/PointCloud2   pclToPclRos(keyframe.pcd_, map_frame)      (utilities.hpp:154-161)
#   /keyframe_pose  geometry_msgs/PoseStamped poseEigToPoseStamped(pose_corrected_eig_)  (utilities.hpp:93-112)
# both stamped with the keyframe's timestamp.  Written and read here without ROS (uncompressed chunks, one per keyframe).
# ----------------------------------------------------------------------------------------------------------------------
import struct as _st

_MD5 = {"sensor_msgs/PointCloud2": "1158d486dd51d683ce2f1be655c3c181", "geometry_msgs/PoseStamped": "d3812c3cbc69362b77dc0b19b345f8f5"}
_HDR_DEF = ("uint32 seq\ntime stamp\nstring frame_id\n")
_SEP = "================================================================================\n"
_DEF = {
    "sensor_msgs/PointCloud2": ("Header header\nuint32 height\nuint32 width\nPointField[] fields\nbool    is_bigendian\nuint32  point_step\n"
                                "uint32  row_step\nuint8[] data\nbool is_dense\n" + _SEP + "MSG: std_msgs/Header\n" + _HDR_DEF + _SEP +
                                "MSG: sensor_msgs/PointField\nuint8 INT8    = 1\nuint8 UINT8   = 2\nuint8 INT16   = 3\nuint8 UINT16  = 4\n"
                                "uint8 INT32   = 5\nuint8 UINT32  = 6\nuint8 FLOAT32 = 7\nuint8 FLOAT64 = 8\nstring name\nuint32 offset\n"
                                "uint8  datatype\nuint32 count\n"),
    "geometry_msgs/PoseStamped": ("Header header\nPose pose\n" + _SEP + "MSG: std_msgs/Header\n" + _HDR_DEF + _SEP +
                                  "MSG: geometry_msgs/Pose\nPoint position\nQuaternion orientation\n" + _SEP +
                                  "MSG: geometry_msgs/Point\nfloat64 x\nfloat64 y\nfloat64 z\n" + _SEP +
                                  "MSG: geometry_msgs/Quaternion\nfloat64 x\nfloat64 y\nfloat64 z\nfloat64 w\n"),
}


def _fields(d):
    out = b""
    for k, v in d.items():
        f = k.encode() + b"=" + v
        out += _st.pack("<I", len(f)) + f
    return out


def _record(header_fields, data):
    h = _fields(header_fields)
    return _st.pack("<I", len(h)) + h + _st.pack("<I", len(data)) + data


def _ros_time(t):
    secs = int(np.floor(t))
    nsecs = int(round((t - secs) * 1e9))
    if nsecs >= 1000000000:
        secs, nsecs = secs + 1, nsecs - 1000000000
    return _st.pack("<II", secs, nsecs)


def _ros_string(s):
    b = s.encode()
    return _st.pack("<I", len(b)) + b


def _rpy_quaternion(R):
    """poseEigToPoseStamped: tf::Matrix3x3::getRPY then tf::createQuaternionFromRPY (utilities.hpp:96-100)."""
    if abs(R[2, 0]) >= 1.0:
        yaw, roll = 0.0, np.arctan2(R[2, 1], R[2, 2])
        pitch = np.pi / 2.0 if R[2, 0] < 0 else -np.pi / 2.0
    else:
        pitch = -np.arcsin(R[2, 0])
        cp = np.cos(pitch)
        roll = np.arctan2(R[2, 1] / cp, R[2, 2] / cp)
        yaw = np.arctan2(R[1, 0] / cp, R[0, 0] / cp)
    hy, hp, hr = yaw / 2.0, pitch / 2.0, roll / 2.0
    cy, sy, cp_, sp, cr, sr = np.cos(hy), np.sin(hy), np.cos(hp), np.sin(hp), np.cos(hr), np.sin(hr)
    return np.array([sr * cp_ * cy - cr * sp * sy, cr * sp * cy + sr * cp_ * sy, cr * cp_ * sy - sr * sp * cy, cr * cp_ * cy + sr * sp * sy])


def _msg_pointcloud2(seq, stamp, frame, pts):
    """pcl::toROSMsg of a pcl::PointCloud<pcl::PointXYZI>: 32-byte records (x y z 1 | intensity pad pad pad)."""
    n = len(pts)
    rec = np.zeros((n, 8), np.float32)
    rec[:, :3] = pts[:, :3]
    rec[:, 3] = 1.0
    rec[:, 4] = pts[:, 3]
    data = rec.tobytes()
    out = _st.pack("<I", seq) + _ros_time(stamp) + _ros_string(frame) + _st.pack("<II", 1, n) + _st.pack("<I", 4)
    for name, off in (("x", 0), ("y", 4), ("z", 8), ("intensity", 16)):
        out += _ros_string(name) + _st.pack("<IBI", off, 7, 1)
    out += _st.pack("<BII", 0, 32, 32 * n) + _st.pack("<I", len(data)) + data + _st.pack("<B", 1)
    return out


def _msg_posestamped(seq, stamp, frame, T):
    q = _rpy_quaternion(T[:3, :3])
    return (_st.pack("<I", seq) + _ros_time(stamp) + _ros_string(frame) + _st.pack("<3d", T[0, 3], T[1, 3], T[2, 3]) +
            _st.pack("<4d", q[0], q[1], q[2], q[3]))


def save_result_bag(path, clouds, poses, stamps, frame="map"):
    """result.bag as FastLioSamQn::~FastLioSamQn writes it (fast_lio_sam_qn.cpp:377-394): per keyframe one /keyframe_pcd and
    one /keyframe_pose message at the keyframe's timestamp."""
    topics = [("/keyframe_pcd", "sensor_msgs/PointCloud2"), ("/keyframe_pose", "geometry_msgs/PoseStamped")]

    def conn_record(cid):
        topic, typ = topics[cid]
        data = _fields({"topic": topic.encode(), "type": typ.encode(), "md5sum": _MD5[typ].encode(), "message_definition": _DEF[typ].encode()})
        return _record({"op": b"\x07", "conn": _st.pack("<I", cid), "topic": topic.encode()}, data)

    body = b""
    chunk_infos = []
    poses = np.asarray(poses, np.float64).reshape(-1, 4, 4)
    for i, (c, T, t) in enumerate(zip(clouds, poses, stamps)):
        chunk = b""
        offsets = {}
        for cid in (0, 1):
            if i == 0:
                chunk += conn_record(cid)  # a connection is announced in the chunk of its first message
            msg = _msg_pointcloud2(i, t, frame, np.asarray(c, np.float32)) if cid == 0 else _msg_posestamped(i, t, frame, T)
            offsets[cid] = len(chunk)
            chunk += _record({"op": b"\x02", "conn": _st.pack("<I", cid), "time": _ros_time(t)}, msg)
        chunk_pos = 4096 + len(body)
        body += _record({"op": b"\x05", "compression": b"none", "size": _st.pack("<I", len(chunk))}, chunk)
        for cid in (0, 1):
            body += _record({"op": b"\x04", "ver": _st.pack("<I", 1), "conn": _st.pack("<I", cid), "count": _st.pack("<I", 1)},
                            _ros_time(t) + _st.pack("<I", offsets[cid]))
        chunk_infos.append((chunk_pos, t))
    index_pos = 4096 + len(body)
    tail = b"".join(conn_record(cid) for cid in (0, 1))
    for pos, t in chunk_infos:
        tail += _record({"op": b"\x06", "ver": _st.pack("<I", 1), "chunk_pos": _st.pack("<Q", pos), "start_time": _ros_time(t),
                         "end_time": _ros_time(t), "count": _st.pack("<I", 2)}, _st.pack("<IIII", 0, 1, 1, 1))
    hdr = _fields({"op": b"\x03", "index_pos": _st.pack("<Q", index_pos), "conn_count": _st.pack("<I", 2),
                   "chunk_count": _st.pack("<I", len(chunk_infos))})
    magic = b"#ROSBAG V2.0\n"
    pad = 4096 - len(magic) - 4 - len(hdr) - 4
    with open(path, "wb") as f:
        f.write(magic + _st.pack("<I", len(hdr)) + hdr + _st.pack("<I", pad) + b" " * pad + body + tail)


def _parse_fields(b):
    out, o = {}, 0
    while o < len(b):
        (n,) = _st.unpack_from("<I", b, o)
        k, _, v = b[o + 4:o + 4 + n].partition(b"=")
        out[k.decode()] = v
        o += 4 + n
    return out


def _records(b, o=0, end=None):
    end = len(b) if end is None else end
    while o < end:
        (hl,) = _st.unpack_from("<I", b, o)
        h = _parse_fields(b[o + 4:o + 4 + hl])
        (dl,) = _st.unpack_from("<I", b, o + 4 + hl)
        yield h, b[o + 8 + hl:o + 8 + hl + dl], o
        o += 8 + hl + dl


def load_result_bag(path):
    """-> dict(clouds, poses, stamps, frame): the keyframes of a result.bag (uncompressed rosbag 2.0), e.g. one written by the
    reference node.  Poses come back through the message's quaternion."""
    with open(path, "rb") as f:
        b = f.read()
    if not b.startswith(b"#ROSBAG V2.0\n"):
        raise ValueError("not a rosbag 2.0 file")
    conns, pcd, pose = {}, {}, {}
    frame = None

    def on_message(h, data):
        nonlocal frame
        topic = conns[_st.unpack("<I", h["conn"])[0]]
        secs, nsecs = _st.unpack("<II", h["time"])
        t = secs + nsecs * 1e-9
        o = 12  # seq + stamp
        (fl,) = _st.unpack_from("<I", data, o)
        frame = data[o + 4:o + 4 + fl].decode()
        o += 4 + fl
        if topic == "/keyframe_pcd":
            height, width, nf = _st.unpack_from("<III", data, o)
            o += 12
            offs = {}
            for _ in range(nf):
                (nl,) = _st.unpack_from("<I", data, o)
                name = data[o + 4:o + 4 + nl].decode()
                off, dt, cnt = _st.unpack_from("<IBI", data, o + 4 + nl)
                offs[name] = (off, dt)
                o += 4 + nl + 9
            _be, step, _row = _st.unpack_from("<BII", data, o)
            o += 9
            (dl,) = _st.unpack_from("<I", data, o)
            raw = np.frombuffer(data, np.uint8, dl, o + 4).reshape(height * width, step)
            out = np.zeros((height * width, 4), np.float32)
            for col, name in enumerate(("x", "y", "z", "intensity")):
                if name in offs:
                    out[:, col] = raw[:, offs[name][0]:offs[name][0] + 4].copy().view(np.float32)[:, 0]
            pcd[t] = out
        elif topic == "/keyframe_pose":
            px, py, pz, qx, qy, qz, qw = _st.unpack_from("<7d", data, o)
            T = np.eye(4)
            T[:3, :3] = _quat_to_rot(np.array([qx, qy, qz, qw]) / np.linalg.norm([qx, qy, qz, qw]))
            T[:3, 3] = (px, py, pz)
            pose[t] = T

    for h, data, _ in _records(b, 13):
        op = h["op"][0]
        if op == 0x05:
            if h["compression"] != b"none":
                raise ValueError("compressed chunks (%s) are not supported" % h["compression"].decode())
            for h2, d2, _ in _records(data):
                if h2["op"][0] == 0x07:
                    conns[_st.unpack("<I", h2["conn"])[0]] = h2["topic"].decode()
                elif h2["op"][0] == 0x02:
                    on_message(h2, d2)
        elif op == 0x07:
            conns[_st.unpack("<I", h["conn"])[0]] = h["topic"].decode()
    stamps = sorted(pcd)
    return dict(clouds=[pcd[t] for t in stamps], poses=np.array([pose[t] for t in stamps]), stamps=np.array(stamps), frame=frame)
