"""Per-role wait profile of the learner's streaming fc1 kernel (fc1_stream_ts_kernel, or fc1_stream_kernel with
PMB_FC1_TS=0), or with --rollout of the rollout step's fc1_stream_kernel (select_actions, 16384 envs).  --obs bf16 feeds
bf16-stored obs (pmb_batch.obs_dtype).  Needs a library built with
PMB_EXTRA_NVCC_FLAGS=-DPMB_FC1_PROFILE python -c 'from pymarl_b200.build import build; build(force=True)'.

    python tools/fc1_role_profile.py [--obs fp32|bf16] [--rollout]"""
import argparse, sys, os, ctypes as C
_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT); sys.path.insert(0, os.path.join(_ROOT, "tests"))
import torch as th
import bench
from cuda_utils import Logger
from pymarl_b200 import le_REGISTRY, mac_REGISTRY, _lib
from pymarl_b200.synthetic import make_scheme, torch_episode_fields
ap = argparse.ArgumentParser()
ap.add_argument("--obs", choices=("fp32", "bf16"), default="fp32")
ap.add_argument("--rollout", action="store_true")
a = ap.parse_args()
shape = bench.SMAC_SHAPES["27m_vs_30m"]
B, T = (16384, 4) if a.rollout else (2048, 180)
dev = th.device("cuda", 0)
args = bench.default_args(shape, mixer="qmix", device="cuda", use_cuda=True, learner_log_interval=10 ** 12, precision="bf16")
th.manual_seed(7)
scheme, groups = make_scheme(shape)
scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
learner = le_REGISTRY["q_learner"](mac, scheme, Logger(), args)
learner.cuda()
fields = torch_episode_fields(shape, B, T, seed=1000, ragged=False, device=dev, with_onehot=False)
if a.obs == "bf16":
    fields["obs"] = fields["obs"].to(th.bfloat16)
batch = bench._DictBatch(fields, B, T)
lib = _lib.lib()
out = (C.c_ulonglong * 16)()


def step(i):
    if a.rollout:
        mac._run_step(batch, 1, epsilon=0.05, seed=1, offset=i, want_actions=True, want_q=False)
    else:
        learner.train(batch, i, 0)


if a.rollout:
    mac.init_hidden(B)
for i in range(2):
    step(i)
lib.pmb_debug_fc1_prof(out, 1)
for i in range(1 if not a.rollout else 20):
    step(3 + i)
lib.pmb_debug_fc1_prof(out, 1)
v = list(out)
n_cta = v[9]
tot = v[8] / n_cta
n_prod = round(v[15] / n_cta)                  # producer warps = staging slots
# (slot, name, warps of the role); per warp: cycles over the kernel's cycles
rows = [(0, "producer: st_empty", n_prod), (10, "producer: descriptors", n_prod), (11, "producer: tables + copies", n_prod),
        (1, "converter: st_full", 8), (6, "converter: load + pack", 8), (7, "converter: store incl. a_free", 8),
        (2, "converter: a_free", 8), (3, "MMA: a_full", 1), (4, "MMA: tempty", 1), (5, "epilogue: tfull", 4),
        (12, "epilogue: x stage free + barrier", 4), (13, "epilogue: work incl. x bulk stores", 4),
        (14, "epilogue: W into TMEM (once)", 4)]
print("obs", a.obs, "rollout" if a.rollout else "learner", "CTAs", n_cta, "cycles per CTA", round(tot), "staging slots", n_prod)
for i, nm, m in rows:
    if v[i]:
        print(f"{nm:38s} {v[i] / n_cta / m / tot * 100:6.1f} % of the kernel time per warp")
