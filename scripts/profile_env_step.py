"""A few eager env steps at [envs] for ncu (-k regex:"post_physics|stack_shift_kernel"): python scripts/profile_env_step.py [envs]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from isaac_b200 import _lib
from isaac_b200.envs.hector_config import HectorCfg
from isaac_b200.envs.hector_env import HectorFreeEnvB200
from isaac_b200.physics import SyntheticPhysics
from isaac_b200.synthetic import make_tape

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
dev = torch.device("cuda:0")
lib = _lib.load(check_device=True)
tape = make_tape(n, 4, seed=1234, fall_prob=0.005, randomize_gains=True)
phys = SyntheticPhysics(n, device=dev)
phys.load_frame(tape.physics[0].to(dev))
env = HectorFreeEnvB200(HectorCfg(), sim_device="cuda:0", physics=phys, statics=tape.statics)
flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
for k in range(3):
    phys.load_frame(tape.physics[k + 1].to(dev))
    flush.zero_()
    torch.cuda.synchronize()
    env.step(tape.noise[k + 1].actions.to(dev))
    torch.cuda.synchronize()
print("done")
