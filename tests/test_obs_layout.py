"""The observation row layout of the CUDA code (ObsLayout, mate_b200/csrc/mate_common.cuh), without a GPU:
tests/native/obs_layout_harness.cu prints the block starts, row widths and the packer's affine partition for the
entity counts of every preset, and they must match mate_b200/constants.py, which follows the reference's format."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from mate_b200 import constants
from mate_b200.config import PRESETS, flatten_config

HERE = os.path.dirname(os.path.abspath(__file__))


def test_layout_matches_constants(tmp_path):
    nvcc = os.environ.get('NVCC') or shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not found')
    exe = str(tmp_path / 'obs_layout_harness')
    subprocess.run([nvcc, '-O2', '-std=c++17', '-o', exe, os.path.join(HERE, 'native', 'obs_layout_harness.cu')],
                   check=True, capture_output=True, timeout=300)
    shapes = sorted({(c['num_cameras'], c['num_targets'], c['num_obstacles'])
                     for c in (flatten_config(cfg) for cfg in PRESETS.values())})
    out = subprocess.run([exe] + [str(n) for shape in shapes for n in shape], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.splitlines()

    nw = constants.NUM_WAREHOUSES
    assert [int(x) for x in lines[0].split()[1:]] == [
        constants.PRESERVED_DIM, 3 + 1, constants.PRESERVED_DIM + constants.TARGET_STATE_DIM_PRIVATE - nw]
    affine = np.cumsum([0, constants.PRESERVED_DIM, constants.TARGET_STATE_DIM_PRIVATE, constants.CAMERA_STATE_DIM_PRIVATE,
                        constants.TARGET_STATE_DIM_PUBLIC + 1, constants.OBSTACLE_STATE_DIM + 1,
                        constants.CAMERA_STATE_DIM_PUBLIC + 1]).tolist()

    assert len(lines) == 1 + len(shapes)
    for shape, line in zip(shapes, lines[1:]):
        head, cam, tgt, aff = [[int(x) for x in part.split()] for part in line.split('|')]
        assert tuple(head) == shape
        cam_idx = constants.camera_observation_indices_of(*shape).tolist()
        tgt_idx = constants.target_observation_indices_of(*shape).tolist()
        assert cam[:6] == cam_idx, shape
        assert tgt[:6] == tgt_idx, shape
        assert cam[6:] == cam_idx[3:], shape   # end of each entity list, from its last entry
        assert tgt[6:] == tgt_idx[3:], shape
        assert aff == affine
