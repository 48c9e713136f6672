"""TEST INFRASTRUCTURE ONLY -- the parity oracle for the STAR hot path.

Nothing in ``star_b200`` (the product) may import this package.  Only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU legs
(``cpu_baseline`` / ``--impl reference``) use it, and only as the checker or
as the timed CPU reference, never as the thing shipped.

Contents
--------
ref_loader.py   loads the UNMODIFIED reference files from /root/reference with
                five import shims (xformers, fairscale, timm, torchsde,
                easydict).  Only works in the build container; the GPU box has
                no /root/reference.
unet_ref.py     CPU/fp32 restatement (plain torch functional ops) of
                ControlledV2VUNet.forward + VideoControlNet.forward, driven by
                a reference-layout state_dict.  Travels to the GPU box.
sampler_ref.py  restatement of noise_schedule / sample_sr / denoise /
                dpmpp_2m_sde with an injectable noise sampler.
kernel_ref.py   per-kernel torch references of every C-ABI entry point
                (what each CUDA kernel must compute, incl. its rounding points).
make_golden.py  runs the real reference here and writes tests/golden/*.
make_golden_reference.py  the same for the tests that compare the CogVideoX path, the UNet restatement
                and the CLI boundary against the reference (CPU cases, and GPU cases on a B200).

Parity status: UNet / sampler restatements are PINNED against the real
reference modules executed in this container (tests/test_oracle_pinning.py,
tests/golden/).  The VAE (diffusers 0.30.0) and CogVideoX (sat 0.4.12) are
un-vendored third-party code that cannot be imported here: parity unpinned.
"""
