"""GPU: closing a generation worker gives back all the device memory it took, so a process that opens and closes
workers (a test session, a server reloading a model) does not grow.

mem_get_info reads the whole device: another process allocating on the same GPU during the test shows up here too.
The bar (16 MB over four cycles) is far below what one leaked RoPE table alone costs per cycle (64 MB)."""
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import ollamamq_b200 as mq  # noqa: E402
from oracle import llama_ref as R  # noqa: E402

MiB = 1 << 20


def _open_close():
    # max_seq 131 072 at head_dim 128: a 64 MB RoPE table beside a 268 MB KV cache
    with mq.Worker(0, mq.model_cfg(R.TINY_LLAMA, max_batch=1, max_seq=131072, max_prefill_tokens=256)):
        pass


def test_open_close_returns_device_memory():
    _open_close()  # warm-up: module loading and the runtime's first-use allocations stay for the process
    torch.cuda.synchronize()
    free_before, _ = torch.cuda.mem_get_info()
    for _ in range(4):
        _open_close()
    torch.cuda.synchronize()
    free_after, _ = torch.cuda.mem_get_info()
    lost = free_before - free_after
    assert lost <= 16 * MiB, f"{lost / MiB:.1f} MB of device memory not returned after 4 open / close cycles"
