"""Ordered reuse of a context's SoA staging: qlb_solve_records unpacks the caller's records into that staging
asynchronously, so a second qlb_solve_records on another stream and a later *_host call must wait for it before they
overwrite the rows."""
import numpy as np
import pytest

from quadruped_locomotion_b200 import capi, synth

pytestmark = pytest.mark.gpu


def test_records_on_two_streams_then_host_call_match_serial_runs(qlb_built):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device")
    B = 200_000   # two chunks of the staging per call
    solver = capi.Solver("quadruped_model")
    recs = [capi.wrench_records(synth.make_states("C5", B, start=s)) for s in (11, 5 * B)]
    st = synth.make_states("C3", B, start=17)
    d_in = [torch.from_numpy(r.view(np.uint8).reshape(-1)).cuda() for r in recs]
    d_out = [torch.zeros(B * capi.RESULT_RECORD_DTYPE.itemsize, dtype=torch.uint8, device="cuda") for _ in recs]

    def records_result(i):
        return d_out[i].cpu().numpy().view(capi.RESULT_RECORD_DTYPE).copy()

    # serial runs
    ref = []
    for i in range(2):
        solver.solve_records(d_in[i], d_out[i], stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        ref.append(records_result(i))
        d_out[i].zero_()
    ref_host = solver.solve_wrench_numpy(st)
    torch.cuda.synchronize()

    # the same three calls with no synchronisation between them
    streams = [torch.cuda.Stream() for _ in range(2)]
    for i in range(2):
        solver.solve_records(d_in[i], d_out[i], stream=streams[i].cuda_stream)
    got_host = solver.solve_wrench_numpy(st)
    torch.cuda.synchronize()
    for i in range(2):
        got = records_result(i)
        assert got.tobytes() == ref[i].tobytes(), f"records call {i}"
    for k in ("grf", "tau", "netwrench", "flags"):
        assert np.array_equal(got_host[k], ref_host[k]), k
    solver.close()
