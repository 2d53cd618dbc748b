"""ROS ingestion (SURVEY.md 8 row f3): the online surface of the reference -- `ROS`, `Sensor`, `Lidar`, `Odometria`
(ICM_SLAM.py:267-449, sensors_definitions.py) -- feeding the same solver, plus an in-process stand-in for the rosbridge
client so that the surface can be exercised (and tested) where roslibpy is not installed.

What the reference does online (sensors.py:16-104): two topic listeners append decoded messages to per-sensor histories; after
every message `principal_callback` aligns the two histories by TIMESTAMP (`Sensor.sort`: message k is the one whose stamp lies
within one sampling period of t0 + k * deltat, searched from a guess that follows the observed message rate) and appends one
column per aligned pair to `mediciones` (B x T), `odometria` (3 x T), `u` (2 x T); a `std_srvs/SetBool` service raises
`iterations_flag`, after which the offline sweeps run on what has arrived.

Here the arrays grow in preallocated host buffers (amortised doubling instead of one np.hstack per message), and the columns
that arrived are handed to the device after every `pump` call (`ROS.feed`): the first through `Engine.load`, later ones through
`Engine.append`, which extracts them on arrival, and pass 0 advances over them (`Engine.pass0_advance`), so `positions` and the
map under construction exist while the robot is still driving, as in the reference.  When the iterations flag is raised,
`Engine.pass0_finish` filters the map built so far and the sweeps start on the data already on the device.  The feeding runs on
the thread that runs `inicializar_online`, never inside a transport callback (a handle is not thread-safe).  `OnlineICM` =
`ICM_ROS` of the reference: the solver façade + this transport.

The fake transport (`FakeRos`, `publish_log`) restates matlab2ros/createbag.py:35-153: `sensor_msgs/LaserScan` and
`nav_msgs/Odometry` dictionaries with a running header (seq, stamp = seq * 0.1 s), delivered to the subscribed callbacks in
process -- optionally with dropped or delayed messages to exercise the re-synchronisation of `Sensor.sort`.
"""
from __future__ import annotations

import math
from copy import deepcopy

import numpy as np

from .icm import ICM_SLAM


# ---- sensors (ICM_SLAM.py:343-449, sensors_definitions.py) ---------------------------------------------------------------
class Sensor:
    """One topic: its decoded message history and the timestamp alignment of ICM_SLAM.py:376-428."""

    def __init__(self, config="", name="name", topic="", topic_msg="", principalCallback=None):
        self.msgs = []
        self.k0 = 0          # index of the last message that was matched
        self.c = 0           # ... and the column it was matched to
        self.t0 = 0.0
        self.config = config
        self.name = name
        self.topic = topic
        self.topic_msg = topic_msg
        self.principalCallback = principalCallback or (lambda: None)
        self.warnings = 0    # messages found out of place or not at all (the reference prints; tests read the count)

    def header_process(self, msg):
        """ICM_SLAM.py:430-442: sequence number and stamp in seconds."""
        st = msg["header"]["stamp"]
        return {"seq": msg["header"].get("seq", 0), "stamp": st["secs"] + st["nsecs"] * 10 ** (-9)}

    def set_t0(self):
        self.t0 = self.msgs[0]["stamp"]

    def subscribe(self, client):
        client.topic(self.topic, self.topic_msg).subscribe(self.callback)

    def callback(self, msg):       # overridden by the concrete sensors
        D = self.header_process(msg)
        D["data"] = None
        self.msgs.append(D)
        self.principalCallback()

    def sort(self, k):
        """The message of column k (stamp within deltat of t0 + k * deltat), ICM_SLAM.py:376-428: first the guess
        ceil(k0 * k / c) that extrapolates the message rate seen so far, then a linear search from the last match.
        Returns (data, True) or (None, False)."""
        ts = self.config.deltat
        now = k * ts + self.t0
        if self.c != 0:
            k1 = int(np.ceil(self.k0 * k / self.c))
            k1 = min(k1, len(self.msgs) - 1)
        else:
            k1 = min(k, len(self.msgs) - 1)
        if abs(self.msgs[k1]["stamp"] - now) < ts:
            self.k0, self.c = k1, k
            return self.msgs[k1]["data"], True
        for i in range(self.k0, len(self.msgs)):
            if abs(self.msgs[i]["stamp"] - now) < ts:
                self.warnings += 1                  # "datos desincronizados, adaptando..."
                self.k0, self.c = i, k
                return self.msgs[i]["data"], True
        self.warnings += 1                          # "no se encuentra la secuencia buscada"
        return None, False


class Lidar(Sensor):
    """sensor_msgs/LaserScan -> one B x 1 column of pre-conditioned ranges (sensors_definitions.py:10-35)."""

    def callback(self, msg):
        D = self.header_process(msg)
        z = np.array([[np.nan if r is None else r for r in msg["ranges"]]], dtype=np.float64)
        z[np.isnan(z)] = self.config.rango_laser_max                                   # :20
        z = np.minimum(z + self.config.radio, self.config.rango_laser_max)              # :21-22
        if z.shape[1] != 180:                                                           # :23-29 (a 181-beam log passes through this too)
            inc = msg["angle_increment"]
            s0 = int((-np.pi / 2 - msg["angle_min"]) / inc)
            step = round((np.pi / 180.0) / inc)
            z = z[:, s0:step * 180:step]
        D["data"] = z.T
        self.msgs.append(D)
        self.principalCallback()


class Odometria(Sensor):
    """nav_msgs/Odometry -> pose (x, y, yaw from the quaternion) and controls (v, w) (sensors_definitions.py:37-74)."""

    def callback(self, msg):
        D = self.header_process(msg)
        p = msg["pose"]["pose"]
        q = p["orientation"]
        yaw = math.atan2(2.0 * (q["w"] * q["z"] + q["x"] * q["y"]), 1.0 - 2.0 * (q["y"] ** 2 + q["z"] ** 2))
        tw = msg["twist"]["twist"]
        D["data"] = {"odo": np.array([[p["position"]["x"], p["position"]["y"], yaw]]).T,
                     "u": np.array([[tw["linear"]["x"], tw["angular"]["z"]]]).T}
        self.msgs.append(D)
        self.principalCallback()


# ---- growing logs ------------------------------------------------------------------------------------------------------------
class _Columns:
    """rows x T array that grows by columns in amortised O(1) (the reference re-allocates with np.hstack per message)."""

    def __init__(self):
        self.buf = None
        self.n = 0

    def append(self, col):
        col = np.asarray(col, dtype=np.float64).reshape(-1)
        if self.buf is None:
            self.buf = np.empty((col.size, 64))
        if self.n == self.buf.shape[1]:
            nb = np.empty((self.buf.shape[0], 2 * self.n))
            nb[:, : self.n] = self.buf[:, : self.n]
            self.buf = nb
        self.buf[:, self.n] = col
        self.n += 1

    def view(self):
        return np.array([]) if self.buf is None else self.buf[:, : self.n]


# ---- the transport (ICM_SLAM.py:267-341) -----------------------------------------------------------------------------------
class ROS:
    """Mixin with the reference's names.  `connect_ros(client)` takes any object with the small client surface used here
    (`topic(name, type).subscribe(cb)`, `service(name, type).advertise(handler)`, `terminate()`, `is_connected`): `FakeRos`
    below, or `RoslibpyClient()` where roslibpy is installed (default when no client is given)."""

    def _ros_init(self, config):
        self.new_data = 0
        self.iterations_flag = False
        self._med, self._odo, self._u = _Columns(), _Columns(), _Columns()
        D = dict(config=config, principalCallback=self.principal_callback)
        self.lidar = Lidar(name="lidar", topic=config.topic_laser, topic_msg=config.topic_laser_msg, **D)
        self.odom = Odometria(name="odometria", topic=config.topic_odometry, topic_msg=config.topic_odometry_msg, **D)
        self.client = None
        self._fed = 0            # aligned columns handed to the solver's engine
        self._walking = False    # pass 0 walks them (False: nothing fed yet, or column 0 has no observation)

    def connect_ros(self, client=None):
        self.client = client if client is not None else RoslibpyClient()
        if not self.client.is_connected:
            self.disconnect_ros()
            raise ConnectionError("no connection to the ROS bridge")
        self.odom.subscribe(self.client)
        self.lidar.subscribe(self.client)
        self.client.service("/icm_slam/iterative_flag", "std_srvs/SetBool").advertise(self.icm_iterations_service)

    def disconnect_ros(self):
        if self.client is not None:
            self.client.terminate()

    def icm_iterations_service(self, request, response):
        """ICM_SLAM.py:292-299: any call raises the flag that ends the online phase."""
        response["success"] = True
        response["message"] = "Working..."
        self.iterations_flag = True
        return True

    def principal_callback(self):
        """ICM_SLAM.py:301-341: append every column for which both sensors have an aligned message."""
        num_msg = min(len(self.odom.msgs), len(self.lidar.msgs))      # (the reference counts the odometry twice; with both sensors
        if num_msg == 0:                                              #  at the same rate the two are equal: this form never indexes
            return                                                    #  past the shorter history)
        num_sensor = self._odo.n
        if num_sensor == 0:
            self.lidar.set_t0()
            self.odom.set_t0()
        for k in range(num_sensor, num_msg):
            laser, ok1 = self.lidar.sort(k)
            aux, ok2 = self.odom.sort(k)
            if not (ok1 and ok2):
                continue
            self._med.append(laser)
            self._odo.append(aux["odo"])
            self._u.append(aux["u"])
            self.new_data += 1
        self.mediciones, self.odometria, self.u = self._med.view(), self._odo.view(), self._u.view()

    def feed(self, engine):
        """Hands every aligned column that arrived since the last call to `engine` -- the first ones through `load` + `extract`,
        later ones through `append` -- and advances pass 0 over them (x0 = odometria[:, 0], sensors.py:61): `positions` is then
        the causal estimate of every column walked (sensors.py:104).  Each column goes to the engine once, in order.  Returns the
        columns fed so far."""
        T = self._u.n                       # (principal_callback appends to the laser log first and to the controls last)
        if T == self._fed:
            return T
        cols = slice(self._fed, T)
        z, odo, u = self._med.buf[:, cols], self._odo.buf[:, cols], self._u.buf[:, cols]
        if self._fed == 0:
            engine.load(z, odo, u, precondition=False)
            engine.extract()
            self.x0 = np.array([odo[:, 0]]).T
            self._walking = engine.pass0_begin(self.x0.reshape(3)) == 0
        else:
            engine.append(z, odo, u)
        self._fed = T
        if self._walking:
            t = engine.pass0_advance()
            self.positions = engine.get_poses()[:, :t]
        return T


class OnlineICM(ICM_SLAM, ROS):
    """`ICM_ROS` of the reference (sensors.py:15-104): the solver with the ROS transport attached."""

    def __init__(self, config, x0=""):
        ICM_SLAM.__init__(self, config, x0)
        self._ros_init(config)
        self.mediciones, self.odometria, self.u = np.array([]), np.array([]), np.array([])

    def inicializar_online(self, client=None, pump=None):
        """sensors.py:51-104.  Connects, lets the messages arrive -- `pump(self)` is called until it returns False or the
        iterations service has been called (a fake publisher delivers its log there; with a real bridge the callbacks run on
        the client's thread and `pump` only has to wait) -- and after every `pump` call feeds what arrived to the engine and
        advances pass 0 over it (`feed`: x0 = odometria[:, 0], :61; `positions` follows).  Then Mapa.filtrar of the map built
        (:99-102): returns (mapa_viejo, positions) as `inicializar` does on the same log."""
        self.connect_ros(client)
        try:
            while pump is not None:
                more = pump(self)
                self.feed(self._engine)
                if not more or self.iterations_flag:
                    break
            self.feed(self._engine)
        finally:
            self.disconnect_ros()
        if self.new_data == 0:
            raise RuntimeError("no aligned laser / odometry message pair arrived")
        self.adopt_engine(self._engine)         # (the engine holds the log: iterar does not upload it again)
        if self._walking:
            xs, mapa = self._engine.pass0_finish()
        else:                                   # an empty first scan: what pass 0 returns then (sensors.py:137-139)
            xs, mapa = self._engine.pass0(self.x0.reshape(3))
        self.mapa_viejo = mapa.copy()
        self.positions = xs.copy()
        self.iterations_flag = True
        return mapa, xs


# ---- clients -----------------------------------------------------------------------------------------------------------------
class RoslibpyClient:
    """The rosbridge client of the reference (ICM_SLAM.py:271-285); needs roslibpy."""

    def __init__(self, host="localhost", port=9090):
        import roslibpy                                       # (absent in this image: FakeRos stands in)
        self._r = roslibpy
        self.c = roslibpy.Ros(host=host, port=port)
        self.c.run()

    @property
    def is_connected(self):
        return self.c.is_connected

    def topic(self, name, typ):
        return self._r.Topic(self.c, name, typ)

    def service(self, name, typ):
        return self._r.Service(self.c, name, typ)

    def terminate(self):
        self.c.terminate()


class _FakeTopic:
    def __init__(self):
        self.subs = []

    def subscribe(self, cb):
        self.subs.append(cb)

    def publish(self, msg):
        for cb in self.subs:
            cb(deepcopy(msg))


class _FakeService:
    def __init__(self):
        self.handler = None

    def advertise(self, handler):
        self.handler = handler

    def call(self, request=None):
        response = {}
        ok = self.handler(request or {"data": True}, response) if self.handler else False
        return ok, response


class FakeRos:
    """In-process stand-in for the rosbridge client: topics deliver synchronously to their subscribers."""

    def __init__(self):
        self.is_connected = True
        self.topics, self.services = {}, {}

    def topic(self, name, typ=""):
        return self.topics.setdefault(name, _FakeTopic())

    def service(self, name, typ=""):
        return self.services.setdefault(name, _FakeService())

    def terminate(self):
        self.is_connected = False


def laser_scan_msg(ranges, seq, dt=0.1):
    """matlab2ros/createbag.py:35-58 + the running header of :108-123 (stamp = seq * dt)."""
    s = seq * dt
    return {"header": {"seq": seq, "stamp": {"secs": int(s), "nsecs": int((s - int(s)) * 10 ** 9)}, "frame_id": "Lidar_horizontal"},
            "angle_min": -np.pi / 2, "angle_max": np.pi / 2, "angle_increment": np.pi / 180, "time_increment": 0.0, "scan_time": 0.0,
            "range_min": 0.5, "range_max": 20.0,
            "ranges": [None if (r is None or (isinstance(r, float) and math.isnan(r))) else float(r) for r in ranges], "intensities": []}


def odometry_msg(odo, vel, seq, dt=0.1):
    """matlab2ros/createbag.py:60-106: yaw -> quaternion (roll = pitch = 0), twist from the controls."""
    s = seq * dt
    yaw = float(odo[2])
    return {"header": {"seq": seq, "stamp": {"secs": int(s), "nsecs": int((s - int(s)) * 10 ** 9)}, "frame_id": "odom_groundtruth"},
            "child_frame_id": "base_link",
            "pose": {"pose": {"position": {"x": float(odo[0]), "y": float(odo[1]), "z": 0.0},
                              "orientation": {"x": 0.0, "y": 0.0, "z": math.sin(yaw / 2.0), "w": math.cos(yaw / 2.0)}}},
            "twist": {"twist": {"linear": {"x": float(vel[0]), "y": 0.0, "z": 0.0}, "angular": {"x": 0.0, "y": 0.0, "z": float(vel[1])}}}}


def publish_log(client, config, ranges, odometry, controls, drop_laser=(), drop_odometry=(), laser_first=True, dt=0.1):
    """Replays a log (raw ranges B x T, odometry 3 x T, controls 2 x T) as the message stream createbag.py produces
    (:124-153).  `drop_*`: time indices whose message of that sensor is lost (the stamps keep running)."""
    lt = client.topic(config.topic_laser, config.topic_laser_msg)
    ot = client.topic(config.topic_odometry, config.topic_odometry_msg)
    T = ranges.shape[1]
    for t in range(T):
        sends = []
        if t not in drop_laser:
            sends.append(lambda t=t: lt.publish(laser_scan_msg(ranges[:, t].tolist(), t, dt)))
        if t not in drop_odometry:
            sends.append(lambda t=t: ot.publish(odometry_msg(odometry[:, t], controls[:, t], t, dt)))
        for f in (sends if laser_first else reversed(sends)):
            f()
    return T
