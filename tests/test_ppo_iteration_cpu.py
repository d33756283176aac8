"""CPU side of kbs_rollout_record and ppo.PpoUpdater.iteration: the ctypes mirror of struct kbs_rollout_record against the
header, the exported symbol, the XLA-FFI handler and jax_ffi wrapper that forward to it, and the updater's public surface."""

import inspect
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_rollout_record_struct_matches_header(lib_built):
    from kbot_joystick_b200 import _lib as L

    hdr = (ROOT / "include" / "kbotstep.h").read_text()
    body = re.search(r"\nstruct kbs_rollout_record \{(.*?)\};", hdr, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [re.sub(r"^(const\s+)?(float|uint8_t)\s*\*\s*", "", d.strip()) for d in body.split(";") if d.strip()]
    assert names == [f[0] for f in L.KbsRolloutRecord._fields_] == ["done_prev", "critic_obs"]
    assert re.search(r"int kbs_rollout_record\(kbs_handle\* h, const kbs_rollout_io\* io, const struct kbs_rollout_record\* rec,",
                     hdr)
    assert int(re.search(r"#define KBS_VERSION (\d+)", hdr).group(1)) == L.VERSION == 101
    assert "kbs_rollout_record" in L.EXPORTS
    assert hasattr(L.load(), "kbs_rollout_record")


def test_rollout_record_ffi_handler_and_wrapper():
    import kbot_joystick_b200.jax_ffi as kf

    cc = (ROOT / "kbot-joystick_b200" / "csrc" / "kbs_xla_ffi.cc").read_text()
    assert kf._TARGETS["kbs_rollout_record"] == "KbsRolloutRecord"
    assert "XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsRolloutRecord, RolloutRecordImpl," in cc
    assert "kbs_rollout_record(H(handle), &io, &rec, n_envs, stream)" in cc
    params = list(inspect.signature(kf.rollout_record).parameters)
    assert params == list(inspect.signature(kf.rollout).parameters)[:-1] + ["done_prev", "n_envs"]


def test_updater_iteration_surface():
    from kbot_joystick_b200.ppo import PpoUpdater

    for name in ("iteration", "capture_iteration"):
        params = inspect.signature(getattr(PpoUpdater, name)).parameters
        assert list(params)[1:] == ["io", "reward_carry", "n_envs", "batch_size", "num_passes", "seed"], name
        assert (params["batch_size"].default, params["num_passes"].default, params["seed"].default) == (512, 3, 0)
