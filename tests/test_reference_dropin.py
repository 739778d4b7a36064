"""Drop-in compatibility with the reference's own classes.  The conversion tests need the reference modules
(oracle/_ref or a reference checkout, see oracle/build_ref.py) and are skipped where they are absent."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import _ref_shim  # noqa: E402


@pytest.fixture(scope="module")
def ref():
    if not _ref_shim.available():
        pytest.skip("reference checkout not present")
    _ref_shim.install()
    import types

    from nerfstudio.fields import neurad_field
    from nerfstudio.model_components import dynamic_actors, ray_samplers

    return types.SimpleNamespace(neurad_field=neurad_field, dynamic_actors=dynamic_actors, ray_samplers=ray_samplers)


def _small(cfg, log2):
    cfg.grid.static.log2_hashmap_size = log2
    return cfg


def test_field_conversion_keeps_names_and_values(ref):
    from neuradar_b200 import plugin

    actors = ref.dynamic_actors.DynamicActors(ref.dynamic_actors.DynamicActorsConfig(), trajectories=[])
    rf = ref.neurad_field.NeuRADField(_small(ref.neurad_field.NeuRADFieldConfig(), 8), actors, static_scale=100.0,
                                      implementation="torch")
    mine = plugin.convert_field(rf)
    ref_sd = rf.state_dict()  # the reference's DynamicActors module rides along, so even its keys line up
    my_sd = mine.state_dict()
    assert sorted(ref_sd.keys()) == sorted(my_sd.keys())
    for k in ref_sd:
        assert torch.equal(ref_sd[k], my_sd[k]), k
    assert mine.hashgrid.static_scale == 100.0
    # the other direction: a checkpoint written by this package loads into the reference module
    assert not rf.load_state_dict(my_sd, strict=False).unexpected_keys

    rp = ref.neurad_field.NeuRADProposalField(_small(ref.neurad_field.NeuRADProposalFieldConfig(), 8), actors, 100.0,
                                              implementation="torch")
    mp = plugin.convert_proposal_field(rp)
    assert sorted(mp.state_dict().keys()) == sorted(rp.state_dict().keys())
    assert torch.equal(mp.density_decoder.weight, rp.density_decoder.weight)


def test_sampler_conversion(ref):
    from neuradar_b200 import plugin

    rs = ref.ray_samplers.ProposalNetworkSampler(
        num_proposal_samples_per_ray=(64, 48), num_nerf_samples_per_ray=48, num_proposal_network_iterations=2,
        single_jitter=True, initial_sampler=ref.ray_samplers.PowerSampler(lambda_=-1.0, scaling=0.1),
        update_sched=lambda x: 0,
    )
    rs.step_cb(7)
    mine = plugin.convert_sampler(rs, -1.0, 0.1)
    assert mine.num_proposal_samples_per_ray == (64, 48) and mine.num_nerf_samples_per_ray == 48
    assert mine.initial_sampler.single_jitter is False and mine.pdf_sampler.single_jitter is True
    assert mine._step == 7 and mine._steps_since_update == 1


def test_nerfacc_compat_installs_when_absent():
    from neuradar_b200 import nerfacc_compat

    for name in ("render_weight_from_alpha", "render_weight_from_density", "accumulate_along_rays", "OccGridEstimator"):
        assert hasattr(nerfacc_compat, name)
