"""CPU (Gloo, world_size 2): the p2p classes keep the reference's contract - context lifecycle, command
broadcast, FIFO ordering through a 2-stage pipeline with results returned to the data rank, tuple payloads,
hooks. The reference's own lifecycle test (`test/comm/p2p/test_context.py:23-40`) is restated first."""
import os
import socket
import threading
import torch
import torch.multiprocessing as mp


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _env(port):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    os.environ['CUDA_VISIBLE_DEVICES'] = ''   # this suite is the Gloo path


def test_context_lifecycle_world1(monkeypatch):
    from pipeedge_b200.comm.p2p import DistP2pContext
    # This test runs in the pytest process: hiding the GPUs here (as `_env` does in the spawned ranks) would leave CUDA
    # initialised without devices for every test after it. A world of one has no data plane, so it needs no hiding.
    monkeypatch.setenv('MASTER_ADDR', '127.0.0.1')
    monkeypatch.setenv('MASTER_PORT', str(_free_port()))
    ctx = DistP2pContext(('gloo',), {'world_size': 1, 'rank': 0}, lambda cmd, tensors: None)
    ctx.init()
    ctx.shutdown()
    with DistP2pContext(('gloo',), {'world_size': 1, 'rank': 0}, lambda cmd, tensors: None):
        pass


def _pipeline_worker(rank, world, port, n_ubatch, out_q):
    _env(port)
    torch.set_num_threads(1)
    from pipeedge_b200.comm.p2p import DistP2pContext, DistP2pPipelineStage
    cmds = []
    stop = threading.Event()

    def handle_cmd(cmd, tensors):
        cmds.append((cmd, [t.tolist() for t in tensors]))
        if cmd == 0:
            stop.set()

    results = []
    done = threading.Event()
    hook_log = []

    def handle_results(payload):
        results.append(payload)
        if len(results) == n_ubatch:
            done.set()

    with DistP2pContext(('gloo',), {'world_size': world, 'rank': rank}, handle_cmd) as ctx:
        if rank == 0:
            ctx.cmd_broadcast(1, (torch.tensor([[1, 4], [5, 8]]), torch.tensor([0, 0]), torch.tensor(7)))
            # rank 0 = data rank + stage 0 (model_cfg.py:141-147): src = last stage, dst = stage 1
            work = lambda x: (x + 1.0, torch.full((x.shape[0], 2), 3, dtype=torch.int32))   # tuple payload
            with DistP2pPipelineStage(1, 1, work, handle_results) as stage:
                stage.register_send_post_hook(lambda tensors, tag: hook_log.append((tag, len(tensors))), ('send',))
                for i in range(n_ubatch):
                    stage.enqueue_tensor(torch.full((2, 3), float(i)))
                assert done.wait(60), "results did not arrive"
                stage.check_workers()
                ctx.cmd_broadcast(0)   # as runtime.py: stop is broadcast before the stage context exits
            out_q.put(('results', [r.tolist() for r in results], hook_log))
        else:
            def work(payload):
                x, meta = payload
                assert meta.dtype == torch.int32 and meta.shape == (2, 2)
                return x * 2.0
            with DistP2pPipelineStage(0, 0, work, None):
                assert stop.wait(60), "stop command did not arrive"
            out_q.put(('cmds', cmds))


def test_two_rank_pipeline_fifo_and_commands():
    ctx = mp.get_context('spawn')
    out_q = ctx.Queue()
    port = _free_port()
    n = 9
    procs = [ctx.Process(target=_pipeline_worker, args=(r, 2, port, n, out_q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(2):
        item = out_q.get(timeout=120)
        got[item[0]] = item[1:]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    results, hook_log = got['results']
    assert len(results) == n
    for i, r in enumerate(results):   # FIFO: result i is (i + 1) * 2 everywhere
        assert r == [[(i + 1) * 2.0] * 3] * 2
    assert hook_log == [('send', 2)] * n
    (cmds,) = got['cmds']
    assert cmds[0] == (1, [[[1, 4], [5, 8]], [0, 0], 7])
    assert cmds[-1][0] == 0


def _ragged_worker(rank, world, port, out_q):
    """Payload layouts that change mid-stream: ragged last micro-batch, a tuple with constant host-side metadata, an
    empty tensor, dtype changes - the envelope protocol resends the full description only when the layout changes and
    hands out the SAME host tensors when their bytes did not change."""
    _env(port)
    torch.set_num_threads(1)
    from pipeedge_b200.comm.p2p import DistP2pContext, DistP2pPipelineStage
    stop = threading.Event()
    done = threading.Event()
    results = []
    meta = torch.tensor([[7, 7]], dtype=torch.int32)          # constant across micro-batches, like the QuantPipe metadata
    first = torch.full((4, 3), 1.0)
    inputs = [first, first, torch.full((2, 3), 3.0),                                          # repeat, ragged tail
              torch.zeros((0, 3)), torch.arange(6, dtype=torch.int64).view(2, 3), torch.full((4, 3), 4.0)]

    def handle_results(payload):
        results.append(payload)
        if len(results) == len(inputs):
            done.set()

    with DistP2pContext(('gloo',), {'world_size': world, 'rank': rank},
                        lambda cmd, tensors: stop.set() if cmd == 0 else None) as ctx:
        if rank == 0:
            with DistP2pPipelineStage(1, 1, lambda x: (x, meta), handle_results) as stage:
                for x in inputs:
                    stage.enqueue_tensor(x)
                assert done.wait(60), "results did not arrive"
                stage.check_workers()
                ctx.cmd_broadcast(0)
            out_q.put(('results', [(str(r.dtype), list(r.shape), r.tolist()) for r in results]))
        else:
            seen_meta = []

            def work(payload):
                x, m = payload
                seen_meta.append(m)
                assert m.dtype == torch.int32 and m.tolist() == [[7, 7]]
                return x + x
            with DistP2pPipelineStage(0, 0, work, None):
                assert stop.wait(60), "stop command did not arrive"
            # a payload made of the very same host tensors is not re-sent: the receiver hands out its objects again
            out_q.put(('meta', len(seen_meta), sum(1 for a, b in zip(seen_meta, seen_meta[1:]) if a is b)))


def test_ragged_and_changing_payload_layouts():
    ctx = mp.get_context('spawn')
    out_q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_ragged_worker, args=(r, 2, port, out_q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(2):
        item = out_q.get(timeout=120)
        got[item[0]] = item[1:]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    (results,) = got['results']
    assert [r[1] for r in results] == [[4, 3], [4, 3], [2, 3], [0, 3], [2, 3], [4, 3]]
    assert results[0][2] == results[1][2] == [[2.0] * 3] * 4 and results[2][2] == [[6.0] * 3] * 2 and results[3][2] == []
    assert results[4][0] == 'torch.int64' and results[4][2] == [[0, 2, 4], [6, 8, 10]]
    assert results[5][0] == 'torch.float32' and results[5][2] == [[8.0] * 3] * 4
    n_meta, n_same = got['meta']
    assert n_meta == 6 and n_same == 1      # payloads 0 and 1 were the same objects on the sender: received once
