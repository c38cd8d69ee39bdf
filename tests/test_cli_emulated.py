"""CPU tier: the product's C ABI layer (csrc/capi.cu) and its `csdr` CLI (host/csdr_cli.c) on top of the EMULATED kernels.

tests/host_shim/emul_build.build_full() compiles every product translation unit for the host under tests/host_shim/cuda_emul.h into one
library with the product's real C ABI and links the unmodified CLI source against it.  The pipe-graph tests of tests/test_gpu_cli.py
then run here, against the unmodified reference CLI (or its recorded outputs), in a container without a GPU: block framing, EOF quirks, preamble, --fifo-less
graphs of the README, and the reference's own binary running on our library through LD_PRELOAD.
Test artefacts only (temporary directory); the product's library still refuses to work without a GPU (tests/test_abi.py).
"""
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests" / "host_shim"))
sys.path.insert(0, str(ROOT / "tests"))
import emul_build  # noqa: E402

pytest.importorskip("torch")
import test_gpu_cli as g  # noqa: E402  (only its helpers and test bodies; its own fixture and gpu mark stay behind)


@pytest.fixture(scope="module")
def clis(tmp_path_factory):
    if not emul_build.available():
        pytest.skip("needs g++ and the CUDA toolkit headers")
    lib, cli = emul_build.build_full_once(tmp_path_factory)
    saved = g.LIB
    g.LIB = lib                                                            # what the LD_PRELOAD test injects into the reference binary
    yield str(cli), str(g.REF) if g.REF.exists() else g.REFERENCE         # without the reference build: its recorded outputs
    g.LIB = saved


test_config1_graph_matches_reference_cli = g.test_config1_graph_matches_reference_cli
test_eof_framing_quirks = g.test_eof_framing_quirks
test_nfm_style_chain = g.test_nfm_style_chain
test_deemphasis_nfm_command = g.test_deemphasis_nfm_command
test_full_nfm_graph_of_the_readme = g.test_full_nfm_graph_of_the_readme
test_shift_addfast_and_decimating_shift_commands = g.test_shift_addfast_and_decimating_shift_commands
test_wfm_graph_of_csdr_fm = g.test_wfm_graph_of_csdr_fm
test_fft_commands = g.test_fft_commands
test_spectrum_and_unroll_commands = g.test_spectrum_and_unroll_commands
test_dynamic_bufsize_preamble = g.test_dynamic_bufsize_preamble
test_reference_binary_runs_on_our_library = g.test_reference_binary_runs_on_our_library

import test_gpu_zz_shift_math as zz  # noqa: E402
test_shift_math_command = zz.test_shift_math_command

import test_gpu_zz_adpcm as za  # noqa: E402
test_adpcm_commands = za.test_adpcm_commands
test_openwebrx_waterfall_chain = za.test_openwebrx_waterfall_chain

import test_gpu_zz_control as zc  # noqa: E402
test_initial_tuning_through_the_control_channel = zc.test_initial_tuning_through_the_control_channel
test_midstream_retune_at_a_known_block = zc.test_midstream_retune_at_a_known_block

import test_gpu_zz_shift_table as zt  # noqa: E402
test_shift_table_command = zt.test_shift_table_command
