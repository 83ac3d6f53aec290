"""The launcher routes of the three replay kernel templates, one row per route (not a test module).

`launch_replay_es` in kfpos_t6.cu, kfpos_k8.cu and kfpos_t9.cu picks one instantiation of t6_replay_kernel,
k8_replay_kernel or t9_replay_kernel from the batch configuration, the range stream and the host flags of
kfpos_api.cu (T9: an IMU event since set_state stays latched; K8 / T9: ml_initial_position keeps the
initialising instantiation while a filter may still be uninitialised).  Every route exists three times: without
per-epoch statistics, with them (ES) and with them and a histogram (ES + EH).

Each row is the template tuple the route reaches, without the ES / EH flags, and a recipe for a small workload
that reaches it.  tests/test_replay_routes_symbols.py checks the table against the kernels the built library
defines; tests/test_gpu_replay_routes.py runs every row and checks with the profiler that the row's kernel ran.
"""
from dataclasses import dataclass
from typing import Tuple

# template parameters in declaration order, ES and EH excluded
TEMPLATE_ARGS = {
    "t6_replay_kernel": ("PME", "LOO", "MT", "SEL", "FMT"),
    "k8_replay_kernel": ("PME", "MT", "SEL", "MLI"),
    "t9_replay_kernel": ("PME", "MT", "IMU", "SEL"),
}
KERNEL = {"T6": "t6_replay_kernel", "K8": "k8_replay_kernel", "T9": "t9_replay_kernel"}
STATS = ((False, False), (True, False), (True, True))  # (ES, EH)


@dataclass(frozen=True)
class Route:
    model: str                 # "T6", "K8" or "T9"
    tup: Tuple                 # the template arguments of KERNEL[model], ES / EH excluded
    m: int = 8                 # anchors
    fmt: str = "i32"           # wire format of the rangings: "f64" (m), "i32" or "u16" (mm)
    pme: bool = False          # per-ranging error estimates
    dtf: bool = False          # per-filter time steps (replay_epochs)
    variant: int = 0           # EKF-side NLOS variant (1: drop the worst, 2: best group)
    loo: bool = False          # T6 leave-one-out (ignore_worst_anchor)
    mli: bool = False          # ml_initial_position, some filters start uninitialised (K8: 2-D mode)
    zero_tz: bool = False      # K8 ml2d_zero_tentative_z
    imu: bool = False          # T9: accelerometer events in the schedule
    big: bool = False          # also run at N = 1000

    @property
    def kernel(self):
        return KERNEL[self.model]

    @property
    def id(self):
        return "%s<%s>" % (self.model, ",".join(str(int(v)) for v in self.tup))

    def symbol(self, es, eh):
        """The demangled kernel name, as nm -C and the profiler print it."""
        return "%s<%s>" % (self.kernel, ", ".join(_arg(v) for v in tuple(self.tup) + (es, eh)))


def _arg(v):
    return ("true" if v else "false") if isinstance(v, bool) else str(v)


T, F = True, False
ROUTES = [
    # T6 <PME, LOO, MT, SEL, FMT>: kfpos_t6.cu launch_replay_es / launch_tuned
    Route("T6", (T, F, 0, T, -1), pme=True, variant=1),
    Route("T6", (F, F, 0, T, -1), variant=2),
    Route("T6", (T, T, 0, F, -1), pme=True, loo=True),
    Route("T6", (F, T, 8, F, -1), loo=True),
    Route("T6", (F, T, 16, F, -1), m=16, loo=True),
    Route("T6", (F, T, 0, F, -1), m=12, loo=True),
    Route("T6", (T, F, 0, F, -1), pme=True),
    Route("T6", (F, F, 4, F, -1), m=4),
    Route("T6", (F, F, 0, F, -1), m=12),
    Route("T6", (F, F, 8, F, 0), fmt="f64", big=True),
    Route("T6", (F, F, 8, F, 1), big=True),
    Route("T6", (F, F, 8, F, 2), fmt="u16", big=True),
    Route("T6", (F, F, 8, F, -1), dtf=True, big=True),
    Route("T6", (F, F, 16, F, 0), m=16, fmt="f64", big=True),
    Route("T6", (F, F, 16, F, 1), m=16, big=True),
    Route("T6", (F, F, 16, F, 2), m=16, fmt="u16", big=True),
    Route("T6", (F, F, 16, F, -1), m=16, dtf=True, big=True),
    # K8 <PME, MT, SEL, MLI>: kfpos_k8.cu launch_replay_es / launch_tuned, make_k8cfg
    Route("K8", (T, 0, T, T), pme=True, variant=1),
    Route("K8", (F, 0, T, T), dtf=True),
    Route("K8", (T, 0, F, F), pme=True),
    Route("K8", (F, 8, F, F), big=True),
    Route("K8", (F, 0, F, F), m=6),
    Route("K8", (T, 0, F, T), pme=True, mli=True),
    Route("K8", (F, 8, F, T), mli=True, big=True),
    Route("K8", (F, 0, F, T), zero_tz=True, mli=True),
    # T9 <PME, MT, IMU, SEL>: kfpos_t9.cu launch_replay_es, run_events (imu_seen, ml_init)
    Route("T9", (T, 0, T, T), pme=True, variant=1),
    Route("T9", (F, 0, T, T), mli=True),
    Route("T9", (T, 0, F, F), pme=True),
    Route("T9", (F, 8, F, F)),
    Route("T9", (F, 0, F, F), m=6),
    Route("T9", (T, 0, T, F), pme=True, imu=True),
    Route("T9", (F, 8, T, F), imu=True),
    Route("T9", (F, 0, T, F), m=6, imu=True),
]
