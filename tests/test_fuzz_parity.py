"""Randomised differential tests (tools/fuzz_parity.py): random cameras, lights and settings on random shader configurations.
(1) the device code compiled for the CPU against the oracle; (2) the oracle against the reference shader compiled as C++, through the sha256 of
its frames stored in tests/golden/ref_fuzz.json (tools/make_ref_golden.py fuzz). Bit for bit. The tool itself runs hundreds of frames
(python tools/fuzz_parity.py --frames 500); these are short samples of it."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import fuzz_parity  # noqa: E402


def test_device_code_matches_the_oracle_on_random_frames():
	mismatches, compared, lit = fuzz_parity.run(frames=24, seed=101, with_reference=False, verbose=False)
	assert compared["device code vs oracle"] >= 18 and lit >= 20
	assert mismatches["device code vs oracle"] == 0 and mismatches["device G-buffer code vs oracle"] == 0 and compared["device G-buffer code vs oracle"] == 24


def test_device_code_matches_the_oracle_on_any_legal_configuration():
	"""Settings the reference was not compiled for here (other strategy / heuristic / biased / vertex count / output stage combinations): run-time parameters for
	both the oracle and the kernels."""
	mismatches, compared, lit = fuzz_parity.run(frames=30, seed=303, with_reference=False, verbose=False, any_config=True, wild=True)
	assert compared["device code vs oracle"] == 30 and lit >= 24
	assert not any(mismatches.values())


def test_oracle_matches_the_reference_shader_on_random_frames():
	with open(os.path.join(ROOT, "tests", "golden", "ref_fuzz.json")) as f:
		golden = json.load(f)
	assert (golden["frames"], golden["seed"]) == (16, 202)
	mismatches, compared, lit = fuzz_parity.run(frames=16, seed=202, with_reference=True, verbose=False, reference_digests=golden["reference"])
	assert compared["reference vs oracle"] == 16 and lit >= 12
	assert not any(mismatches.values())
