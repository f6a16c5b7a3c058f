"""Signature with the reference's interface (bls_py/signature.py:8-130)."""
from . import ec
from .util import GROUP_ORDER


class Signature:
    SIGNATURE_SIZE = 96

    def __init__(self, value, aggregation_info=None):
        self.value = value                      # ec.Point on G2
        self.aggregation_info = aggregation_info

    @staticmethod
    def from_bytes(buffer, aggregation_info=None, check_subgroup=False):
        """check_subgroup=True: ValueError also for a point outside G2 (the reference accepts it)"""
        return Signature(ec.point_from_bytes(bytes(buffer), True, check_subgroup), aggregation_info)

    @staticmethod
    def from_bytes_batch(buffers, check_subgroup=False):
        """many signatures decoded in one GPU call (no aggregation info attached)"""
        return [Signature(p) for p in ec.points_from_bytes(buffers, True, check_subgroup)]

    @staticmethod
    def from_g2(g2_el, aggregation_info=None):
        return Signature(g2_el, aggregation_info)

    def divide_by(self, divisor_signatures):
        """Quotient of an aggregate by some of its constituents (signature.py:44-103): every
        (message hash, key) pair of a divisor must be in this signature's tree, and the ratio
        dividend / divisor exponent must be the same for all pairs of one divisor.  The curve
        work -- one scalar multiplication per divisor and one sum -- is two batched GPU calls."""
        remove, points, scalars = [], [], []
        for div in divisor_signatures:
            info = div.aggregation_info
            if len(info.public_keys) != len(info.message_hashes):
                raise Exception("Invalid aggregation info")
            quotient = None
            for key in zip(info.message_hashes, info.public_keys):
                divisor = info.tree[key]
                if key not in self.aggregation_info.tree:
                    raise Exception("Signature is not a subset")
                q = self.aggregation_info.tree[key] * pow(divisor, -1, GROUP_ORDER) % GROUP_ORDER
                if quotient is None:
                    quotient = q
                elif q != quotient:
                    raise Exception("Cannot divide by aggregate signature, msg/pk pairs are not unique")
                remove.append(key)
            if quotient is not None:
                points.append(div.value)
                scalars.append(-quotient % GROUP_ORDER)
        value = ec.sum_points([self.value] + ec.scalar_mul_many(points, scalars, True), True)
        info = self.aggregation_info.copy()
        for key in remove:
            info.tree.pop(key, None)
        keys = sorted(info.tree.keys())
        info.message_hashes = [k[0] for k in keys]
        info.public_keys = [k[1] for k in keys]
        return Signature(value, info)

    def set_aggregation_info(self, aggregation_info):
        self.aggregation_info = aggregation_info

    def get_aggregation_info(self):
        return self.aggregation_info

    def serialize(self):
        return self.value.serialize()

    def size(self):
        return self.SIGNATURE_SIZE

    def __eq__(self, other):
        return self.serialize() == other.serialize()

    def __hash__(self):
        return int.from_bytes(self.serialize(), "big")

    def __lt__(self, other):
        return self.serialize() < other.serialize()

    def __repr__(self):
        return "Signature(%s)" % self.serialize().hex()

    __str__ = __repr__
