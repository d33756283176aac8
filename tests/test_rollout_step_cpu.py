"""CPU side of the online rollout: the ctypes mirrors of kbs_step_state, kbs_step_carry and kbs_step_io against the header,
the exported symbols, the kernel id of the step's record pass, and PpoUpdater's online surface."""

import inspect
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def fields_of(hdr: str, name: str) -> list:
    body = re.search(r"typedef struct " + name + r" \{(.*?)\} " + name + ";", hdr, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [d.strip().split()[-1].lstrip("*") for d in body.split(";") if d.strip()]


def test_step_structs_match_header(lib_built):
    from kbot_joystick_b200 import _lib as L

    hdr = (ROOT / "include" / "kbotstep.h").read_text()
    assert fields_of(hdr, "kbs_step_state") == [f[0] for f in L.KbsStepState._fields_]
    assert fields_of(hdr, "kbs_step_carry") == [f[0] for f in L.KbsStepCarry._fields_]
    assert fields_of(hdr, "kbs_step_io") == [f[0] for f in L.KbsStepIO._fields_]
    lib = L.load()
    for name in ("kbs_step_state_bytes", "kbs_step_state_load", "kbs_step_state_store", "kbs_step_state_rewind",
                 "kbs_rollout_step"):
        assert name in L.EXPORTS and hasattr(lib, name), name
    assert int(re.search(r"#define KBS_NUM_KERNEL_IDS (\d+)", hdr).group(1)) == L.NUM_KERNEL_IDS
    assert b"step_record_kernel" in [lib.kbs_kernel_name(i) for i in range(L.NUM_KERNEL_IDS)]
    assert int(re.search(r"#define KBS_STATUS_STEP_RANGE (0x[0-9a-f]+)", hdr).group(1), 16) == L.STATUS_STEP_RANGE


def test_updater_online_surface():
    from kbot_joystick_b200.ppo import PpoUpdater

    assert list(inspect.signature(PpoUpdater.begin_iteration).parameters)[1:] == ["io", "n_envs"]
    assert list(inspect.signature(PpoUpdater.step).parameters)[1:] == ["io_t"]
    assert list(inspect.signature(PpoUpdater.capture_step).parameters)[1:] == ["io_t"]
    params = inspect.signature(PpoUpdater.end_iteration).parameters
    assert list(params)[1:] == ["reward_carry", "n_envs", "batch_size", "num_passes", "seed"]
