"""The CUDA engine against the reference ITSELF, on the same box in the same test: the reference's unmodified
election / replication / commit code (oracle/_ref/libref_stack.so on the verbs shim, N host processes) and the GPU
engine (through the C ABI) are fed the same request stream; the logs they leave behind must be identical --
leader copy: every byte, reply bytes included; follower copies: every byte outside reply[0..12] (H5 mask,
SURVEY.md s8c) plus the follower's own ack byte (I7).  Leader index and term are whatever the reference's
election produced.  The reference's side is the recording of these runs in tests/golden/refstack_runs_golden.json
(tests/golden/gen_refstack_golden.py), which tests/test_oracle_vs_refstack.py also checks the oracle against."""
import pytest

import orc as O
import refstack as R
from refgold import recorded, sha

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]


@pytest.fixture(scope="module")
def eng():
    import __graft_entry__ as g
    g.build()
    import apus_b200
    if apus_b200.lib().apus_device_count() < 1:
        pytest.fail("no CUDA device visible on a gpu-marked test")
    return apus_b200


@pytest.mark.parametrize("n,nconn,nreq,plen", [(3, 2, 300, 64), (5, 3, 200, 128), (3, 1, 120, -3000), (7, 4, 400, 64)])
def test_engine_log_equals_reference_log(eng, n, nconn, nreq, plen):
    rr = recorded("refstack_runs_golden.json")[f"log_equals/{n}/{nconn}/{nreq}/{plen}"]
    lead, term = rr["leader"], rr["term"]
    nd = eng.lib().apus_device_count()
    with eng.Group(n, devices=[i % nd for i in range(n)], leader=lead, term=term, log_size=O.LOG_SIZE) as g:
        g.prologue()
        g.submit_stream(R.expected_stream(lead, nconn, nreq, plen))
        g.run()
        end = rr["results"][lead]["offsets"]["end"]
        for i in range(n):
            ro, eo = rr["results"][i]["offsets"], g.replicas[i].offsets()
            assert (eo["end"], eo["commit"], eo["head"], eo["len"]) == (ro["end"], ro["commit"], ro["head"], ro["len"]), (i, eo, ro)
            if i == lead:
                assert eo["tail"] == ro["tail"]
            got, want = g.replicas[i].image(0, end), rr["images"][i]
            assert want["len"] == end
            ents = O.walk_entries(got, 0, end, O.LOG_SIZE)
            assert len(ents) == rr["entries"]
            if i != lead:
                for off, _ in ents:
                    assert got[off + 28 + i] == 1
                assert all(bytes.fromhex(k)[1 + i] == 1 for k in want["stamps"])
                assert sha(O.mask_replies(got, ents)) == want["masked_sha"], f"replica {i} (leader {lead}, term {term})"
            else:
                assert sha(got) == want["sha"], f"replica {i} (leader {lead}, term {term})"
        assert g.leader.committed() == len(ents)
