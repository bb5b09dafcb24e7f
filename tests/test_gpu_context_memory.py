"""A closed Context gives back the device memory it held: every work buffer, YART_FLAG_NEXT_EVENT's path state included."""
import pytest

pytestmark = pytest.mark.gpu

GIB = 1 << 30


def _next_event_render(yart, w, h, spp):
    """One render of cornell-box with next-event estimation in a fresh context, closed afterwards; returns its stats."""
    ctx = yart.Context(0)
    try:
        preset = yart.ScenePreset("cornell-box", seed=1)
        ctx.set_scene(preset)
        _, st = ctx.render(preset.camera(w, h), w, h, 0, spp, max_depth=2, seed=1, batch_spp=spp,
                           flags=yart.FLAG_NEXT_EVENT)
        return st
    finally:
        ctx.close()


def test_closing_a_context_frees_its_next_event_state(yart):
    """1024 x 1024 pixels x 16 samples in one batch: 16 Mi paths in flight hold 1.27 GB of next-event state (76 B a
    path) besides the path state.  Three such contexts, each closed, leave free memory where it was."""
    import torch
    _next_event_render(yart, 64, 64, 1)  # module loading and other once-per-process device allocations
    torch.cuda.synchronize()
    free_before, _ = torch.cuda.mem_get_info(0)
    for _ in range(3):
        st = _next_event_render(yart, 1024, 1024, 16)
        assert st.paths == 1024 * 1024 * 16
    free_after, _ = torch.cuda.mem_get_info(0)
    assert free_before - free_after < GIB, "closed contexts kept %.2f GiB" % ((free_before - free_after) / GIB)
