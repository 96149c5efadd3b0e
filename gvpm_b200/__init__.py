"""gvpm_b200 — B200-native (sm_100a CUDA) density-estimation gather of the gvpm / sppm integrators.

Only what the hot path needs: csrc/ (kernels + the C ABI of include/gvpm_b200.h), the host-side
mirror of the reference's gather drivers (host.py, host/), the flattened record containers and the
synthetic-input generator.  There is no CPU fallback: see _native.load_lib().
"""
from . import _native
from .records import (BeamSet, PlaneSet, PhotonSet, RaySet, VpmSampleSet, synth_beams, synth_planes, bre_radius, make_config, make_medium, synth_occluders,
                      synth_photons, synth_rays, synth_vpm_samples, box_scene_default, pinhole_camera,
                      lookat_camera, box_scene_as_mesh)

__all__ = ["_native", "PhotonSet", "RaySet", "bre_radius", "make_config", "make_medium",
           "synth_occluders", "synth_photons", "synth_rays", "VpmSampleSet", "synth_vpm_samples",
           "BeamSet", "PlaneSet", "synth_beams", "synth_planes", "box_scene_default", "pinhole_camera",
           "lookat_camera", "box_scene_as_mesh"]
