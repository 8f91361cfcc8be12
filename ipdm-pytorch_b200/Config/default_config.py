"""Options of the IPDM denoiser: same flag names, defaults and merge rules as the reference's
Config/default_config.py (default_cfg :7-172, cfg_load :176-185, load_option :188-194).

The flags are declared from one table instead of ~70 add_argument calls.  Reference quirks kept on
purpose: `type=bool` flags are truthy for any non-empty string; a JSON overlay never overrides a
flag that was given on the command line; `cfg_load` only merges keys that already exist and prints
the reference's "no key names ..." line otherwise.  Additive keys of this build: `precision`
("tf32" | "fp32" | "bf16"), `noise_seed`, `cuda_graph`, `simulate_low_dose` (the test loop makes
its low-dose inputs from the full-dose data at `dose` instead of reading them) and the settings of
the `convertor="SART"` convertor, `sart_iterations` (sweeps), `sart_subsets` (S, divides 2000) and
`sart_relaxation` (lambda in (0, 2)); their defaults reproduce the reference.  The reference's `ntv` is read by
`convertor="SART"`: the number of TV steps after every sweep (SART-TV; 0, the default, is plain SART), with `tv_alpha` (step
fraction of the sweep's change), `tv_eps` (TV smoothing, 1/cm) and `sart_init` ("zero" | "fbp": the start image).
`convertor="PWLS"` (penalised weighted least squares by ordered-subset SQS) reads `sart_iterations`, `sart_subsets`, `sart_init`
and `dose` (the weights are the rays' inverse variances at that dose) and its own `pwls_beta` (penalty weight) and `pwls_delta`
(edge scale of the hyperbola penalty, 1/cm); it ignores `sart_relaxation` and the TV options.
"""
import argparse
import json
import sys

# (name, type, default, nargs)
_FLAGS = [
    # train / test
    ("save_freq", int, 10000, None), ("batch_size", int, 4, None), ("test_batch_size", int, 1, None),
    ("max_epochs", int, 300, None), ("init_lr", float, 2e-4, None), ("test_numbers", int, 50, None),
    ("mode", str, "train_img", None), ("run_name", str, "default", None), ("model_name", str, "IPDM", None),
    ("device", str, "cuda:0", None), ("convertor", str, "TV", None), ("load_option_path", str, None, None),
    ("load_img_model_path", str, None, None), ("load_proj_model_path", str, None, None),
    ("resume_epochs_proj", int, 0, None), ("resume_epochs_img", int, 0, None), ("display_result", bool, False, None),
    ("test_result_data_save", bool, False, None), ("benchmark_test", bool, False, None),
    ("metrics", str, ["psnr", "ssim", "fsim", "vif", "nqm"], "+"), ("fbp_sharpen", bool, False, None), ("ntv", int, 0, None),
    ("normal", bool, False, None), ("ultra_img_denoise", bool, True, None),
    # image-domain model
    ("in_channels_img", int, 1, None), ("out_channels_img", int, 1, None), ("model_channels_img", int, 64, None),
    ("attention_resolutions_img", int, [16], "+"), ("channel_mult_img", float, [1, 1, 2, 2, 4, 4], "+"),
    ("timesteps_img", int, 1000, None), ("partial_timesteps_img", int, 50, None), ("schedule_power_img", float, 1, None),
    ("clip_img", bool, True, None), ("save_states_img", bool, False, None), ("lambda_ratio_img", float, 5, None),
    ("t_start_img", int, None, "+"), ("eta_img", float, 0.5, None), ("constant_guidance_img", float, None, None),
    ("kernel_size_img", int, 4, None), ("amplitude_img", float, 20, None), ("ddim_timesteps_img", int, [1, 2, 2], "+"),
    ("sample_method_img", str, "dense", None), ("save_it_state_img", bool, False, None),
    # projection-domain model
    ("in_channels_proj", int, 1, None), ("out_channels_proj", int, 1, None), ("model_channels_proj", int, 64, None),
    ("attention_resolutions_proj", int, [32], "+"), ("channel_mult_proj", float, [1 / 64, 2 / 64, 4 / 64, 2, 2, 4, 4], "+"),
    ("timesteps_proj", int, 1000, None), ("partial_timesteps_proj", int, 50, None), ("schedule_power_proj", float, 1, None),
    ("clip_proj", bool, False, None), ("lambda_ratio_proj", float, 5, None), ("t_start_proj", int, None, "+"),
    ("eta_proj", float, 0.4, None), ("constant_guidance_proj", float, None, None), ("kernel_size_proj", int, 4, None),
    ("amplitude_proj", float, 5, None), ("ddim_timesteps_proj", int, [1, 2, 2], "+"), ("sample_method_proj", str, "dense", None),
    ("save_it_state_proj", bool, False, None),
    # dataset
    ("data_type", str, "siemens", None), ("train_dataset_path_FD_img", str, None, None),
    ("train_dataset_path_LD_img", str, None, None), ("train_dataset_path_FD_proj", str, None, None),
    ("train_dataset_path_LD_proj", str, None, None), ("test_dataset_path_FD_img", str, None, None),
    ("test_dataset_path_LD_img", str, None, None), ("test_dataset_path_FD_proj", str, None, None),
    ("test_dataset_path_LD_proj", str, None, None), ("num_workers", int, 4, None), ("patch", int, [512, 512], "+"),
    ("patch_per_image", int, 4, None), ("dose", float, 0.25, None),
    # additive (B200 build)
    ("precision", str, "tf32", None), ("noise_seed", int, 0, None), ("cuda_graph", bool, False, None),
    ("simulate_low_dose", bool, False, None), ("sart_iterations", int, 5, None), ("sart_subsets", int, 100, None),
    ("sart_relaxation", float, 1.0, None), ("tv_alpha", float, 0.2, None), ("tv_eps", float, 1e-4, None), ("sart_init", str, "zero", None),
    ("pwls_beta", float, 1e6, None), ("pwls_delta", float, 0.0002, None),
]


def default_cfg(argv=None):
    parser = argparse.ArgumentParser('Default arguments for training of different domain denoiser')
    for name, typ, default, nargs in _FLAGS:
        kw = dict(type=typ, default=default)
        if nargs:
            kw["nargs"] = nargs
        parser.add_argument('--' + name, **kw)
    argv = sys.argv[1:] if argv is None else argv
    opt = parser.parse_args(argv)
    given = [a[2:] for a in argv if "--" in a]
    if opt.load_option_path is not None:
        print("options are loading...")
        print("loading cfg except {}".format(given))
        load_option(opt, opt.load_option_path, given)
        print("options were loaded successfully!")
    return opt


def cfg_load(new_cfg, old_cfg):
    """Merge `new_cfg` into `old_cfg`, known keys only (nested dicts recurse)."""
    for key, val in new_cfg.items():
        if isinstance(val, dict):
            cfg_load(val, old_cfg[key])
        elif key in old_cfg.keys():
            old_cfg[key] = val
        else:
            print(f"no key names {key} in config\n")


def load_option(opt, load_path, exception):
    with open(load_path, 'r') as f:
        loaded = json.load(f)
    for key in exception:
        loaded.pop(key, None)
    cfg_load(loaded, opt.__dict__)
