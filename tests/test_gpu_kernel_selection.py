"""GPU tests of the step-kernel selection (run with -m gpu on a B200): for every kernel choice, on RGB and symbolic-only
handles of the lean (three-action) and the seven-action configuration, at batch sizes on both sides of every threshold
of the launch policy, the kernel that `step` and `policy_step` launch -- recorded with torch.profiler -- is the one
`step_kernel()` names, and that name is the one the documented table (merlin_set_kernel_choice) gives.  bench.py reports
the label as "kernel" and looks the measured DRAM traffic up by it."""
from __future__ import annotations

import re

import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# Batch sizes N = k x SMs + d (the device's SM count, read in the test): both sides of each threshold -- symbolic-only
# warp <= 2048, RGB warp <= 24 576, tile<16> from SMs x 4 x 16 envs, group size G = the largest of 32 / 16 / 8 with
# N / G >= 8 x SMs.
SIZES = [(0, 1), (0, 2048), (0, 2049), (0, 24576), (0, 24577), (64, -1), (64, 0), (128, -1), (128, 0), (256, -1),
         (256, 0)]


def _expected_label(choice, n, rgb, lean, sms):
    if choice == 0:
        choice = (2 if n <= 24576 else 3) if rgb else (2 if n <= 2048 else 5)
    if choice == 1:
        g = next((g for g in (32, 16, 8) if n // g >= 8 * sms), 4)
        return f"merlin::env_kernel<{g},true>"
    if choice == 3:
        return f"merlin::env_kernel_tile<{16 if n >= sms * 4 * 16 else 8},true>"
    if choice == 7 and not (lean and rgb):
        choice = 2
    return {2: "merlin::env_kernel_warp<true>", 4: "merlin::env_kernel_tile_tma<true>",
            5: "merlin::env_kernel_sym<true>", 6: "merlin::env_kernel_ordered<true>",
            7: "merlin::env_kernel_quad<true>"}[choice]


def _label_key(label):
    """(base name, first template argument or None) of a step_kernel() label such as merlin::env_kernel_tile<16,true>:
    only the group and tile labels carry one (G or T)."""
    base, args = re.fullmatch(r"(merlin::\w+)<(.*)>", label).groups()
    first = args.split(",")[0]
    return base, first if first.isdigit() else None


def _launched_key(name):
    """(base name, first template argument) of a launched kernel, from its demangled or mangled name."""
    m = re.search(r"(merlin::\w+)<\s*([^,>]+)", name)
    if m:
        return m.group(1), m.group(2).strip()
    m = re.search(r"_ZN6merlin(\d+)", name)
    rest = name[m.end():]
    ident = rest[:int(m.group(1))]
    arg = re.match(r"IL[ib](\d+)E", rest[len(ident):])
    return "merlin::" + ident, arg.group(1)


@pytest.fixture(scope="module")
def pool():
    from merlin_b200 import layouts
    return layouts.generate("mediumhard", 16, range(4200, 4264))


@pytest.mark.parametrize("rgb", [True, False], ids=["rgb", "symbolic_only"])
@pytest.mark.parametrize("n_actions", [3, 7], ids=["lean", "seven_actions"])
@pytest.mark.parametrize("k,d", SIZES, ids=[f"{k}sms{d:+d}" if k else str(d) for k, d in SIZES])
def test_step_kernel_label_names_the_launched_kernel(pool, rgb, n_actions, k, d):
    from merlin_b200 import BatchedMerlinEnv
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N = k * sms + d
    cells, agent = pool
    env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, device=DEV, n_actions=n_actions, want_rgb=rgb)
    env.reset()
    actions = torch.randint(0, n_actions, (N,), device=DEV)
    io = env.make_policy_io(torch.randn((N, n_actions), device=DEV))
    labels = []
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for choice in range(8):
            env.set_kernel_choice(choice)
            labels.append(env.step_kernel())
            env.step(actions)
            env.policy_step(io)
        torch.cuda.synchronize()
    env.close()
    kernels = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA and "merlin" in e.name),
                     key=lambda e: e.time_range.start)
    names = [e.name for e in kernels]
    assert len(names) == 16, names   # one step and one policy step per choice, one launch each
    for choice, label in enumerate(labels):
        assert label == _expected_label(choice, N, rgb, n_actions == 3, sms), choice
        base, size = _label_key(label)
        for name in names[2 * choice:2 * choice + 2]:
            launched_base, first_arg = _launched_key(name)
            assert launched_base == base, (choice, label, name)
            if size is not None:
                assert first_arg == size, (choice, label, name)
