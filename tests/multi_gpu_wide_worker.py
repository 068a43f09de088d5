"""
torchrun worker: multi_gpu_worker.py's two-rank epoch against the multi-rank oracle, with a Box action space of
PPOAF_MG_ACT_DIM dimensions (default 100), so the Gaussian head runs the wide loss kernel and its d(log_std) peer
mirrors.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import multi_gpu_worker  # noqa: E402
from ppo_and_friends_b200 import synthetic  # noqa: E402

_make_rollout = synthetic.make_rollout


def _wide_rollout(**kw):
    return _make_rollout(**dict(kw, act_dim=int(os.environ.get("PPOAF_MG_ACT_DIM", "100"))))


if __name__ == "__main__":
    synthetic.make_rollout = _wide_rollout       # read by multi_gpu_worker.main() at call time
    multi_gpu_worker.main()
