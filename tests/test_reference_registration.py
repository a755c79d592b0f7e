"""Drop-in check against MAC-VO's own registry and config specs, recorded from the MAC-VO tree in
tests/golden/macvo_registry.pt (tests/golden/make_golden_macvo.py): for each module of MACVO_Performant.yaml that a B200 class
replaces, the interface MAC-VO files it under, the keys its `is_valid_config` demands and the YAML's args. Each B200 class
must be found by name under the interface of that name, accept the same args (on a CUDA device) through the
interface-level validator `MACVO.is_valid_config` calls (Odometry/MACVO.py:137-156), require every key the replaced class
requires and reject an excess key like it."""
from types import SimpleNamespace as NS

import pytest

B200 = {"frontend": "B200_FlowFormerCovFrontend", "keypoint": "B200_CovAwareSelector_NoDepth",
        "mappoint": "B200_MappingPointSelector", "cov": "B200_MatchCovariance", "optimizer": "B200_TwoFrame_PGO"}


def test_plugins_register_into_macvo_registry(golden):
    from macvo_b200 import plugins as P
    ref = golden("macvo_registry.pt")
    assert set(ref) == set(B200)
    for role, name in B200.items():
        r, cls = ref[role], getattr(P, name)
        iface = next(c for c in cls.__mro__ if c.__name__ == r["interface"])
        assert iface.get_class(name) is cls, (role, r["interface"])
        args = dict(r["args"])
        if "device" in args:
            args["device"] = "cuda"
        if role == "optimizer":
            args["parallel"] = False            # the B200 optimiser's asynchrony is its CUDA stream, not a spawned process
        iface.is_valid_config(NS(type=name, args=NS(**args)))
        for key in r["spec_keys"]:
            with pytest.raises(KeyError):
                cls.is_valid_config(NS(**{k: v for k, v in args.items() if k != key}))
        assert r["excess_rejected"]
        with pytest.raises(KeyError):
            iface.is_valid_config(NS(type=name, args=NS(**args, extra=1)))
    with pytest.raises(ValueError):
        P.B200_MatchCovariance(NS(device="cpu", kernel_size=31, match_cov_default=0.25, min_depth_cov=0.05, min_flow_cov=0.25))


def test_local_interfaces_registry_and_config_spec():
    from types import SimpleNamespace as NS
    from macvo_b200 import interfaces as I
    from macvo_b200 import plugins as P
    if not P._REF:
        assert I.IFrontend.get_class("B200_FlowFormerCovFrontend") is P.B200_FlowFormerCovFrontend
        I.IKeypointSelector.is_valid_config(NS(type="B200_MappingPointSelector",
                                               args=NS(max_depth=5.0, max_depth_cov=0.005, mask_width=32)))
        with pytest.raises(KeyError):
            P.B200_MappingPointSelector.is_valid_config(NS(max_depth=5.0, max_depth_cov=0.005))
        with pytest.raises(KeyError):
            I.IFrontend.get_class("NoSuchFrontend")
    with pytest.raises(ValueError):
        P.B200_CovAwareSelector_NoDepth(NS(device="cpu", kernel_size=7, mask_width=32, max_match_cov=100.0))
