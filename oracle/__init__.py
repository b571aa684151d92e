"""ORACLE -- test infrastructure only (never imported by detectorch_b200/)."""
import os

# torch-CPU results depend, in the last bits, on the instruction set ATen / oneDNN / MKL pick and on the thread count.  The bit-exact
# fixture of the reference detector's outputs (tests/golden/net_golden_r50fpn_128x160.npz) is produced and checked under this
# environment (AVX2 code paths, one thread), so that it holds on any x86-64 host with AVX2.  It must be set before torch starts.
CPU_BITWISE_ENV = {"ATEN_CPU_CAPABILITY": "avx2", "ONEDNN_MAX_CPU_ISA": "AVX2", "MKL_CBWR": "AVX2", "OMP_NUM_THREADS": "1", "MKL_NUM_THREADS": "1"}


def usable_cpus():
    """Host threads this process may really use: the scheduler affinity mask, capped by the cgroup CPU quota (cpu.max) when there is one.
    os.cpu_count() alone counts every core of the machine, and a torch thread pool of that size inside a smaller cgroup quota runs an
    order of magnitude slower than a right-sized one (the 12x swing of the round-1 cpu_baseline)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)
