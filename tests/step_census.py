"""One GanTrainer step with recording wrappers around ``unet_bssfp_b200.ops`` functions (test plumbing only).

The exact-kernel suites rerun what a real training step issues, at its real shapes, instead of a hand-kept list:
``run_step`` builds the generator and discriminator, wraps the named ops for the duration of one step and restores
them afterwards."""
import pytest
import torch

DEV = "cuda"


def run_step(modality, batch, size, wrappers):
    """Run one ``GanTrainer.step`` (seeded networks and inputs) with ``ops.<name>`` replaced by ``make(original)`` for
    each ``name: make`` of ``wrappers``; the wrappers record what they see and call the original."""
    import unet_bssfp_b200 as ub
    from unet_bssfp_b200 import ops
    from unet_bssfp_b200.train_step import GanTrainer
    cin = 24 if modality == "bssfp" else 6
    with pytest.MonkeyPatch.context() as mp:
        for name, make in wrappers.items():
            mp.setattr(ops, name, make(getattr(ops, name)))
        torch.manual_seed(0)
        g, d = ub.Generator(modality).to(DEV), ub.Discriminator(modality).to(DEV)
        tr = GanTrainer(g, d)
        torch.manual_seed(1)
        x = torch.rand(batch, cin, size, size, size, device=DEV)
        y = torch.rand(batch, 6, size, size, size, device=DEV)
        tr.step(x, y)
        torch.cuda.synchronize()
        del tr, g, d, x, y
    torch.cuda.empty_cache()
