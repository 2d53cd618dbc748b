"""ROS ingestion feeding the solver's engine (ROS.feed, CPU only): every aligned column is handed over exactly once and in order --
the first ones through load + extract, later ones through append -- with lost and late messages, and pass 0 advances after every
feed that brought columns.  A stub stands in for the engine; the run through the real one is in test_online_append.py."""
import numpy as np

from icm_slam_b200 import ros_ingest as ri
from icm_slam_b200.config import ConfigICM

from helpers import CONFIG_ROS


class Ingest(ri.ROS):
    """the transport alone (no solver, no device)"""

    def __init__(self, config):
        self._ros_init(config)
        self.mediciones, self.odometria, self.u = np.array([]), np.array([]), np.array([])
        self.positions = None


class StubEngine:
    def __init__(self):
        self.calls = []
        self.z, self.odo, self.u = [], [], []
        self.T = 0

    def _take(self, z, odo, u):
        assert z.shape[1] == odo.shape[1] == u.shape[1] > 0
        self.z.append(np.array(z)); self.odo.append(np.array(odo)); self.u.append(np.array(u))
        self.T += z.shape[1]

    def load(self, z, odo, u, precondition=False):
        assert not self.calls and precondition is False
        self.calls.append("load")
        self._take(z, odo, u)

    def extract(self):
        self.calls.append("extract")

    def append(self, z, odo, u):
        assert self.calls[:2] == ["load", "extract"]
        self.calls.append("append")
        self._take(z, odo, u)

    def pass0_begin(self, x0):
        self.calls.append("begin")
        self.x0 = np.array(x0)
        return 0

    def pass0_advance(self):
        self.calls.append("advance")
        return self.T

    def get_poses(self):
        return np.tile(np.arange(self.T, dtype=np.float64), (3, 1))


def _log(T, B=181, seed=9):
    rng = np.random.default_rng(seed)
    raw = rng.uniform(0.6, 12.0, (B, T))
    odo = np.stack([np.cumsum(rng.normal(0, 0.1, T)), np.cumsum(rng.normal(0, 0.1, T)), rng.uniform(-3, 3, T)])
    u = np.stack([rng.uniform(0, 1, T), rng.normal(0, 0.3, T)])
    return raw, odo, u


def test_every_aligned_column_reaches_the_engine_once_in_order():
    cfg = ConfigICM.from_values(**dict(CONFIG_ROS, topic_laser="/scan", topic_laser_msg="sensor_msgs/LaserScan", topic_odometry="/odom",
                                       topic_odometry_msg="nav_msgs/Odometry"))
    T = 150
    raw, odo, u = _log(T)
    node, client, eng = Ingest(cfg), ri.FakeRos(), StubEngine()
    node.connect_ros(client)
    lt, ot = client.topic(cfg.topic_laser), client.topic(cfg.topic_odometry)
    late = {}                           # laser messages that arrive after the odometry of the next step
    t, k, feeds = 0, 0, 0
    while t < T:
        t1 = min(T, t + [1, 7, 50, 3][k % 4])
        for s in range(t, t1):
            if s in late:
                lt.publish(late.pop(s))
            m = ri.laser_scan_msg(raw[:, s].tolist(), s)
            if s in (20, 95):
                pass                                  # lost
            elif s in (40, 41, 120):
                late[s + 2] = m
            else:
                lt.publish(m)
            if s not in (61,):                        # one odometry message lost
                ot.publish(ri.odometry_msg(odo[:, s], u[:, s], s))
        n_before = len(eng.calls)
        node.feed(eng)
        if node.new_data > 0 and len(eng.calls) > n_before:
            feeds += 1
            assert eng.calls[-1] == "advance"
            assert node.positions.shape == (3, node.new_data)
        t, k = t1, k + 1
    for m in late.values():
        lt.publish(m)
    node.feed(eng)
    node.feed(eng)                                    # nothing new: nothing handed over
    assert node.lidar.warnings > 0
    Ta = node.new_data
    assert 0 < Ta <= T and eng.T == Ta
    assert np.array_equal(np.concatenate(eng.z, axis=1), node.mediciones)
    assert np.array_equal(np.concatenate(eng.odo, axis=1), node.odometria)
    assert np.array_equal(np.concatenate(eng.u, axis=1), node.u)
    assert eng.calls[:3] == ["load", "extract", "begin"]
    assert eng.calls.count("load") == 1 and eng.calls.count("append") == len(eng.z) - 1 >= 10
    assert eng.calls.count("advance") == len(eng.z) == feeds + (1 if len(eng.z) > feeds else 0)
    assert np.array_equal(eng.x0, node.odometria[:, 0])
    assert np.array_equal(node.x0[:, 0], node.odometria[:, 0])
