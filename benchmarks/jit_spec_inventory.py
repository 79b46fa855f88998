#!/usr/bin/env python
"""Which runtime specialisation imx_jit_compile_check builds, per preset, kind, variant, batch size and tuning switch.  Needs no
GPU.  One JSON line per case: the cubin cache filename the build wrote, or the error the check returned.

The filename is a hash of the build's full specification (kernel names and every -D define, in order) and the embedded
kernel sources, so two library builds with the same kernel sources specialise a case identically exactly when they print the
same filename for it.  Compare the output of two builds with `diff`."""
import argparse
import ctypes
import json
import os
import sys
import tempfile
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from marl_for_im_b200 import _lib, presets  # noqa: E402
from marl_for_im_b200.envs import ENV_CLASSES  # noqa: E402

SERIAL_KINDS, DIV_KINDS = ("IM", "MAIM"), ("IM_div", "MAIM_div")
SWITCHES = [{}, {"IMX_STEP_ET": "0"}, {"IMX_STEP_ET": "1"}, {"IMX_STEP_ET_THREADS": "64"}, {"IMX_ROLLOUT_ET": "0"},
            {"IMX_L2_HINTS": "0"}, {"IMX_L2_HINTS": "1"}, {"IMX_L2_HINTS": "2"}, {"IMX_ACT_PREFETCH": "0"}]


def cases(envs):
    for preset in sorted(presets.PRESETS):
        kinds = DIV_KINDS if preset.startswith("div") else SERIAL_KINDS
        for kind in kinds:
            for n in envs:
                for variant in range(5):
                    for sw in SWITCHES:
                        yield preset, kind, n, variant, sw


def run(case):
    preset, kind, n, variant, sw = case
    out = {"preset": preset, "kind": kind, "num_envs": n, "variant": variant, "switches": sw}
    with tempfile.TemporaryDirectory() as cache:        # a fresh cache: the one file that appears is this case's build
        env = {k: os.environ.get(k) for k in list(sw) + ["IMX_CACHE_DIR"]}
        os.environ.update(sw, IMX_CACHE_DIR=cache)
        try:
            c = ENV_CLASSES[kind](dict(presets.PRESETS[preset](), num_envs=n, _config_only=True)).imx_config
            lib = _lib.load()
            rc = lib.imx_jit_compile_check(ctypes.byref(c), variant, None, 0)
            if rc > 0:
                out["cubin"] = sorted(f for f in os.listdir(cache) if f.endswith("_sm100a.cubin"))
            else:
                out["error"] = [rc, lib.imx_last_error().decode()]
        except Exception as exc:                         # a config the env class refuses for this kind
            out["error"] = [None, f"{type(exc).__name__}: {exc}"]
        finally:
            for k, v in env.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="65536,1048576")
    ap.add_argument("--jobs", type=int, default=os.cpu_count() or 4)
    args = ap.parse_args()
    envs = [int(x) for x in args.envs.split(",")]
    with ProcessPoolExecutor(max_workers=args.jobs) as pool:
        for out in pool.map(run, list(cases(envs)), chunksize=4):
            print(json.dumps(out, sort_keys=True), flush=True)


if __name__ == "__main__":
    main()
