"""CPU fp32 oracle for the multi-frame ESRGAN hot path -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this package; nothing under satlas_super_resolution_b200/ does (the product path has no CPU fallback).

What it restates (plain torch fp32 on the CPU, functional style over a state_dict):
  nets.py    SSR_RRDBNet.forward            /root/reference/ssr/archs/rrdbnet_arch.py:37-44,63-68,116-137
             SSR_UNetDiscriminatorSN.forward /root/reference/ssr/archs/discriminator_arch.py:42-71
             torch.nn.utils.spectral_norm (legacy hook API, 1 power iteration, eps 1e-12)
  losses.py  basicsr==1.4.2 L1Loss / GANLoss(vanilla) / PerceptualLoss(VGG19) / USMSharp -- basicsr is a
             requirements.txt:1 dependency that is NOT vendored under /root/reference and not installed
             here; restated from its published algorithm (SURVEY.md appendix A.3/A.4) and anchored on the
             reference call sites ssr/models/ssr_esrgan_model.py:31,109,148,154,182,218,224.
  step.py    SSRESRGANModel.feed_data / optimize_parameters  ssr/models/ssr_esrgan_model.py:104-233

Pinning: the reference ships no tests, golden vectors or fixtures for this path (SURVEY.md section 4,
8c), so parity is pinned against the reference ITSELF run in the build container: make_golden.py imports
the unmodified reference nn.Modules from /root/reference (through ref_shim.py, which only stubs the
absent basicsr/kornia imports) and writes tests/golden/*.pt; tests/test_oracle.py checks nets.py against
those files (make_golden_ref.py records the remaining reference results the tests compare with).  The basicsr-side pieces
(losses, USM, Adam/EMA wiring) have no runnable reference here: they are "parity unpinned" by the
reference and are cross-checked against the torch / torchvision / cv2 primitives they wrap.
"""
