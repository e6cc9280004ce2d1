"""Small case for compute-sanitizer --leak-check full: weight stores on every path.

On each path (exact, exact + BatchNorm, bf16, split, ResNet) it creates and destroys a context that never uses an opponent, and one that
snapshots its networks into the opponent store (mz_snapshot_opponent) and plays one MZ_OPP_NETWORK arena game.  Without the sanitizer it
still reports, from a probe context's mz_device_info (cudaMemGetInfo), the device memory each mz_create takes and what is left after each
mz_destroy; run it twice and the second pass shows whether anything stays behind.  Free bytes are device-wide: on a shared GPU they are
indicative."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from muzero_jl_b200 import capi

PATHS = {
    "exact": lambda: capi.default_config(),
    "exact_bn": lambda: capi.default_config(use_batch_norm=1),
    "bf16": lambda: capi.default_config(nn_mode=capi.NN_BF16_TC),
    "split": lambda: capi.default_config(nn_mode=capi.NN_SPLIT_MMA),
    "resnet": lambda: capi.resnet_config(),
}

probe = capi.Context(capi.default_config(num_slots=1, replay_buffer_size=1))


def free():
    return probe.device_info()["free_bytes"]


out = {}
for rnd in range(2):
    for name, make in PATHS.items():
        f0 = free()
        ctx = capi.Context(make())
        f1 = free()
        ctx.close()
        f2 = free()
        ctx = capi.Context(make())
        ctx.init_weights(5)
        ctx.snapshot_opponent()
        r = ctx.arena(0, 1, capi.OPP_NETWORK, 1, 0.0)
        assert r["wins"] + r["draws"] + r["losses"] == 1
        ctx.close()
        f3 = free()
        out["%s/%d" % (name, rnd)] = dict(create_bytes=f0 - f1, left_after_destroy=f0 - f2, left_after_opponent=f0 - f3)
probe.close()
print(json.dumps(out, indent=1))
print("sanitize wstore ok")
