"""configs[0]: ray.util.collective API, world_size=2, gloo backend on CPU (plumbing, no GPU).

Ported from the reference's single_node_cpu_tests (python/ray/util/collective/tests/
single_node_cpu_tests/test_{allreduce,allgather,reducescatter,broadcast,reduce,sendrecv,basic_apis}.py):
same known-answer values, same error expectations.  The API layer under test is
ant_ray_b200.collective (GroupManager, init/destroy, validation); the arithmetic is real gloo via
the oracle package's restated TorchGLOOGroup.
"""
import numpy as np
import pytest
import torch

from mini_actor import get
from workers import create_collective_workers

from ant_ray_b200.types import Backend, ReduceOp


@pytest.fixture
def workers(store_dir):
    made = []

    def make(n=2, group_name="default"):
        actors = create_collective_workers(n, group_name, "gloo", store_dir)
        made.extend(actors)
        return actors

    yield make
    for a in made:
        a.kill()


@pytest.mark.parametrize("group_name", ["default", "test", "123?34!"])
def test_allreduce_different_name(workers, group_name):
    actors = workers(2, group_name)
    results = get([a.do_allreduce.remote(group_name) for a in actors])
    for r in results:
        assert (r == np.ones((10,), dtype=np.float32) * 2).all()


@pytest.mark.parametrize("array_size", [2, 2**5, 2**10, 2**15, 2**20])
def test_allreduce_different_array_size(workers, array_size):
    actors = workers()
    get([a.set_buffer.remote(np.ones(array_size, dtype=np.float32)) for a in actors])
    results = get([a.do_allreduce.remote() for a in actors])
    for r in results:
        assert (r == np.ones((array_size,), dtype=np.float32) * 2).all()


def test_allreduce_destroy_and_reinit(workers):
    actors = workers()
    results = get([a.do_allreduce.remote() for a in actors])
    assert (results[0] == 2).all()
    get([a.destroy_group.remote() for a in actors])
    with pytest.raises(RuntimeError):
        get([a.do_allreduce.remote() for a in actors])
    get([a.init_group.remote(2, i, "gloo", "default") for i, a in enumerate(actors)])
    results = get([a.do_allreduce.remote() for a in actors])
    for r in results:
        assert (r == np.ones((10,), dtype=np.float32) * 4).all()


def test_allreduce_multiple_group(workers, num_groups=4):
    actors = workers()
    for g in range(1, num_groups):
        get([a.init_group.remote(2, i, "gloo", str(g)) for i, a in enumerate(actors)])
    for i in range(num_groups):
        name = "default" if i == 0 else str(i)
        results = get([a.do_allreduce.remote(name) for a in actors])
        assert (results[0] == np.ones((10,), dtype=np.float32) * (2 ** (i + 1))).all()


def test_allreduce_different_op(workers):
    actors = workers()
    expect = {ReduceOp.PRODUCT: 6, ReduceOp.MIN: 2, ReduceOp.MAX: 3}
    for op, val in expect.items():
        get([a.set_buffer.remote(np.ones(10, dtype=np.float32) * (i + 2)) for i, a in enumerate(actors)])
        results = get([a.do_allreduce.remote(op=op) for a in actors])
        for r in results:
            assert (r == np.ones((10,), dtype=np.float32) * val).all()


@pytest.mark.parametrize("dtype", [np.uint8, np.float16, np.float32, np.float64])
def test_allreduce_different_dtype(workers, dtype):
    actors = workers()
    get([a.set_buffer.remote(np.ones(10, dtype=dtype)) for a in actors])
    results = get([a.do_allreduce.remote() for a in actors])
    for r in results:
        assert (r == np.ones((10,), dtype=dtype) * 2).all()


def test_allreduce_torch_numpy_mixed(workers):
    actors = workers()
    get([actors[0].set_buffer.remote(torch.ones(10)), actors[1].set_buffer.remote(np.ones(10, dtype=np.float32))])
    results = get([a.do_allreduce.remote() for a in actors])
    assert (results[0] == torch.ones(10) * 2).all()
    assert (results[1] == np.ones(10, dtype=np.float32) * 2).all()


@pytest.mark.parametrize("shape", [10, [2, 2], [5, 5, 5]])
def test_allgather_different_shape(workers, shape):
    actors = workers()
    for i, a in enumerate(actors):
        get(a.set_buffer.remote(np.ones(shape, dtype=np.float32) * (i + 1)))
        get(a.set_list_buffer.remote([np.ones(shape, dtype=np.float32) for _ in range(2)]))
    results = get([a.do_allgather.remote() for a in actors])
    for i in range(2):
        for j in range(2):
            assert (results[i][j] == np.ones(shape, dtype=np.float32) * (j + 1)).all()


@pytest.mark.parametrize("length", [0, 1, 3])
def test_allgather_unmatched_list_length(workers, length):
    actors = workers()
    get(actors[0].set_list_buffer.remote([np.ones(10, dtype=np.float32) for _ in range(length)]))
    with pytest.raises(RuntimeError):
        get([a.do_allgather.remote() for a in actors[:1]])


def test_reducescatter(workers):
    actors = workers()
    results = get([a.do_reducescatter.remote() for a in actors])
    for r in results:
        assert (r == np.ones((10,), dtype=np.float32) * 2).all()


@pytest.mark.parametrize("src_rank", [0, 1])
def test_broadcast(workers, src_rank):
    actors = workers()
    get([a.set_buffer.remote(np.ones(10, dtype=np.float32) * (i + 2)) for i, a in enumerate(actors)])
    results = get([a.do_broadcast.remote(src_rank=src_rank) for a in actors])
    for r in results:
        assert (r == np.ones((10,), dtype=np.float32) * (src_rank + 2)).all()


def test_broadcast_invalid_rank(workers):
    actors = workers()
    with pytest.raises(ValueError):
        get([a.do_broadcast.remote(src_rank=3) for a in actors])


@pytest.mark.parametrize("dst_rank", [0, 1])
def test_reduce_leaves_non_root_untouched(workers, dst_rank):
    actors = workers()
    results = get([a.do_reduce.remote(dst_rank=dst_rank) for a in actors])
    for i, r in enumerate(results):
        expect = 2 if i == dst_rank else 1
        assert (r == np.ones((10,), dtype=np.float32) * expect).all()


@pytest.mark.parametrize("shape", [[10], [5, 9, 10, 85]])
def test_sendrecv(workers, shape):
    actors = workers()
    get([a.set_buffer.remote(np.ones(shape, dtype=np.float32) * (i + 1)) for i, a in enumerate(actors)])
    refs = [actors[0].do_send.remote(dst_rank=1), actors[1].do_recv.remote(src_rank=0)]
    results = get(refs)
    assert (results[1] == np.ones(shape, dtype=np.float32)).all()


def test_send_to_self_raises(workers):
    actors = workers()
    with pytest.raises(RuntimeError):
        get(actors[0].do_send.remote(dst_rank=0))


def test_basic_apis(workers):
    actors = workers()
    assert get([a.report_rank.remote() for a in actors]) == [0, 1]
    assert get([a.report_world_size.remote() for a in actors]) == [2, 2]
    assert get([a.report_rank.remote("nope") for a in actors]) == [-1, -1]
    assert get(actors[0].report_is_group_initialized.remote()) is True
    assert get(actors[0].report_is_group_initialized.remote("nope")) is False
    with pytest.raises(RuntimeError):  # initialising the same group twice
        get(actors[0].init_group.remote(2, 0, "gloo", "default"))
    assert get(actors[0].report_gloo_availability.remote()) is True
    # the B200 backend is available exactly when the built library has a CUDA device to run on
    assert get(actors[0].report_nccl_availability.remote()) is torch.cuda.is_available()
    if torch.cuda.is_available():  # the group is declared; its communicator is built by the first collective
        get(actors[0].init_group.remote(2, 0, Backend.B200, "gpu_group"))
        assert get(actors[0].report_is_group_initialized.remote("gpu_group")) is True
    else:  # no CUDA device: refused, there is no CPU fallback
        with pytest.raises(RuntimeError):
            get(actors[0].init_group.remote(2, 0, Backend.B200, "gpu_group"))


def test_backend_names():
    assert Backend("nccl") == Backend.B200 == Backend("b200")
    assert Backend("torch_gloo") == Backend.GLOO == Backend("gloo")
    with pytest.raises(ValueError):
        Backend("mpi")
