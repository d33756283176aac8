"""CPU side of the online rollout's physics sub-steps: the ctypes mirrors of kbs_actuator_state and kbs_substep_io against the
header, the exported symbols, the kernel's profiler name, the range status bit, and PpoUpdater's sub-step surface."""

import inspect
import re
from pathlib import Path

from test_rollout_step_cpu import fields_of

ROOT = Path(__file__).resolve().parent.parent


def test_substep_structs_match_header(lib_built):
    from kbot_joystick_b200 import _lib as L

    hdr = (ROOT / "include" / "kbotstep.h").read_text()
    assert fields_of(hdr, "kbs_actuator_state") == [f[0] for f in L.KbsActuatorState._fields_]
    assert fields_of(hdr, "kbs_substep_io") == [f[0] for f in L.KbsSubstepIO._fields_]
    assert dict(L.KbsSubstepIO._fields_)["episode"] is L.KbsEpisodeView
    lib = L.load()
    for name in ("kbs_actuator_state_bytes", "kbs_actuator_state_load", "kbs_actuator_state_store", "kbs_actuator_substep"):
        assert name in L.EXPORTS and hasattr(lib, name), name
    assert int(re.search(r"#define KBS_NUM_KERNEL_IDS (\d+)", hdr).group(1)) == L.NUM_KERNEL_IDS == 26
    names = [lib.kbs_kernel_name(i).decode() for i in range(L.NUM_KERNEL_IDS)]
    assert "actuator_substep_kernel" in names and "?" not in names
    assert int(re.search(r"#define KBS_STATUS_SUBSTEP_RANGE (0x[0-9a-f]+)", hdr).group(1), 16) == L.STATUS_SUBSTEP_RANGE == 0x400


def test_updater_substep_surface():
    from kbot_joystick_b200.engine import KbotStep
    from kbot_joystick_b200.ppo import PpoUpdater

    for fn in (PpoUpdater.substep, PpoUpdater.capture_substep):
        params = inspect.signature(fn).parameters
        assert list(params)[1:] == ["io_k", "n_substeps", "sub_dt", "drop_prob"]
        assert {k: (params[k].kind, params[k].default) for k in ("n_substeps", "sub_dt", "drop_prob")} == {
            "n_substeps": (inspect.Parameter.KEYWORD_ONLY, 5), "sub_dt": (inspect.Parameter.KEYWORD_ONLY, 0.004),
            "drop_prob": (inspect.Parameter.KEYWORD_ONLY, 0.05)}
    assert list(inspect.signature(KbotStep.actuator_state).parameters)[1:] == ["n_envs", "n_substeps", "prev_action"]
    assert list(inspect.signature(KbotStep.actuator_substep).parameters)[1:] == ["st", "ast", "io_k"]
