"""The backend interface of plonk.keygen / plonk.create_proof (plonk.BACKEND_METHODS, plonk.BACKEND_ATTRIBUTES): every backend
states all of it, the list is exactly what the two functions read from their backend argument, and the sharded backend
picks its quotient path by its number of ranks."""
import ast
import inspect

import pytest

import plonk_model as VM
from util import pm


@pytest.fixture(scope="module")
def PL():
    import __graft_entry__ as ge
    ge.load_package()
    from tiny_ram_halo2_b200 import plonk
    return plonk


def test_every_backend_has_every_method(PL):
    from tiny_ram_halo2_b200.sharded_backend import ShardedGpuBackend
    for cls in (VM.PythonBackend, PL.GpuBackend, ShardedGpuBackend):
        missing = [m for m in PL.BACKEND_METHODS if not callable(getattr(cls, m, None))]
        assert not missing, f"{cls.__name__} lacks {missing}"
        assert isinstance(cls.leaves_are_coefficients, bool)
    assert PL.GpuBackend.leaves_are_coefficients and not VM.PythonBackend.leaves_are_coefficients
    be = VM.PythonBackend(pm.Vesta, 3, 3)
    assert all(hasattr(be, a) for a in PL.BACKEND_ATTRIBUTES)


def test_the_interface_is_what_keygen_and_create_proof_read(PL):
    names = {"B", "backend"}
    reads = set()
    for fn in (PL.keygen, PL.create_proof):
        for node in ast.walk(ast.parse(inspect.getsource(fn))):
            if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id in names:
                reads.add(node.attr)
            if isinstance(node, ast.Call) and isinstance(node.func, ast.Name) and node.func.id in ("hasattr", "getattr"):
                assert not (node.args and isinstance(node.args[0], ast.Name) and node.args[0].id in names), "a capability probe"
    assert set(PL.BACKEND_ATTRIBUTES) == {"n", "p", "q", "k", "j", "extended_k", "omega", "delta", "leaves_are_coefficients"}
    assert len(set(PL.BACKEND_METHODS)) == len(PL.BACKEND_METHODS)
    assert reads == set(PL.BACKEND_METHODS) | set(PL.BACKEND_ATTRIBUTES)


def test_sharded_backend_chooses_its_quotient_by_rank_count(PL):
    """ShardedGpuBackend.quotient_pieces: one rank takes GpuBackend's parts by degree; several take the cached whole program, or
    build_h's Ast when the cache refuses, into the row-sliced quotient()"""
    from types import SimpleNamespace
    from tiny_ram_halo2_b200.sharded_backend import ShardedGpuBackend
    calls = []

    class Fake(ShardedGpuBackend):
        def __init__(self, world, cached):
            self.world, self.cached = world, cached

        def quotient_program(self, pk, build_h, challenges, n_perm_columns):
            calls.append(("program", challenges, n_perm_columns))
            return self.cached

        def quotient(self, prog, leaves):
            calls.append(("whole", prog, leaves))
            return "pieces"

        def quotient_part_programs(self, pk, build_parts, challenges, n_perm_columns):
            return [(ncos, "prog%d" % ncos, keys) for ncos, _, keys in build_parts(*challenges)]

        def quotient_parts(self, parts):
            calls.append(("parts", parts))
            return "pieces"

    pk = SimpleNamespace(vk=SimpleNamespace(cs=SimpleNamespace(permutation=[("advice", 0)] * 3)))
    ch = (1, 2, 3, 4)
    build_h = lambda *c: ("ast", ["a", "b"])
    build_parts = lambda *c: [(1, "ast1", ["a"]), (3, "ast3", ["a", "b"])]
    for world, cached, want in [
            (2, ("cached", ["b"]), [("program", ch, 3), ("whole", "cached", ["B"])]),
            (4, None, [("program", ch, 3), ("whole", "ast", ["A", "B"])]),
            (1, ("cached", ["b"]), [("parts", [(1, "prog1", ["A"]), (3, "prog3", ["A", "B"])])])]:
        calls.clear()
        assert Fake(world, cached).quotient_pieces(pk, ch, build_h, build_parts, str.upper) == "pieces"
        assert calls == want
