"""A small run of every kernel of libewk.so:

    python profiles/tools/sanitize_workload.py [group ...]

The workloads are the groups of tests/test_gpu_poison.py (WORKLOADS), which together launch every __global__ kernel and
template instance of csrc/; each group's docstring names what it reaches.  The memory check itself is
`pytest -m gpu tests/test_gpu_poison.py tests/test_gpu_buffer_edges.py` (DESIGN.md §7: compute-sanitizer is closed on
the GPUs this project is measured on)."""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))


def main(groups):
    from test_gpu_poison import WORKLOADS, run_workload
    for g in groups or list(WORKLOADS):
        run_workload(g, None)
        print(f"{g}: done")
    print("sanitize workload done")


if __name__ == "__main__":
    main(sys.argv[1:])
