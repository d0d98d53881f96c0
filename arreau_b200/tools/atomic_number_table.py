"""Mirror of diffusion/tools/atomic_number_table.py (the part the sampling / checkpoint path touches)."""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

# element symbols by atomic number (the reference uses pymatgen's Element(symbol).number, tools/atomic_number_table.py:88)
_SYMBOLS = ("H He Li Be B C N O F Ne Na Mg Al Si P S Cl Ar K Ca Sc Ti V Cr Mn Fe Co Ni Cu Zn Ga Ge As Se Br Kr Rb Sr Y Zr "
            "Nb Mo Tc Ru Rh Pd Ag Cd In Sn Sb Te I Xe Cs Ba La Ce Pr Nd Pm Sm Eu Gd Tb Dy Ho Er Tm Yb Lu Hf Ta W Re Os Ir "
            "Pt Au Hg Tl Pb Bi Po At Rn Fr Ra Ac Th Pa U Np Pu Am Cm Bk Cf Es Fm Md No Lr").split()
ATOMIC_NUMBER = {s: i + 1 for i, s in enumerate(_SYMBOLS)}

# standard atomic weights (IUPAC, amu) of Z = 1..103, in _SYMBOLS order; for elements without stable isotopes the mass
# number of the longest-lived isotope, as periodic tables print it in brackets
ATOMIC_MASS = (
    1.008, 4.002602, 6.94, 9.0121831, 10.81, 12.011, 14.007, 15.999, 18.998403163, 20.1797,
    22.98976928, 24.305, 26.9815385, 28.085, 30.973761998, 32.06, 35.45, 39.948, 39.0983, 40.078,
    44.955908, 47.867, 50.9415, 51.9961, 54.938044, 55.845, 58.933194, 58.6934, 63.546, 65.38,
    69.723, 72.630, 74.921595, 78.971, 79.904, 83.798, 85.4678, 87.62, 88.90584, 91.224,
    92.90637, 95.95, 98.0, 101.07, 102.90550, 106.42, 107.8682, 112.414, 114.818, 118.710,
    121.760, 127.60, 126.90447, 131.293, 132.90545196, 137.327, 138.90547, 140.116, 140.90766, 144.242,
    145.0, 150.36, 151.964, 157.25, 158.92535, 162.500, 164.93033, 167.259, 168.93422, 173.045,
    174.9668, 178.49, 180.94788, 183.84, 186.207, 190.23, 192.217, 195.084, 196.966569, 200.592,
    204.38, 207.2, 208.98040, 209.0, 210.0, 222.0, 223.0, 226.0, 227.0, 232.0377,
    231.03588, 238.02891, 237.0, 244.0, 243.0, 247.0, 247.0, 251.0, 252.0, 257.0,
    258.0, 259.0, 262.0)


class AtomicNumberTable:
    """tools/atomic_number_table.py:7-26."""
    MASK_ATOMIC_NUMBER = 2001

    def __init__(self, zs: Sequence[int]):
        self.zs = list(zs)

    def __len__(self) -> int:
        return len(self.zs)

    def __str__(self):
        return f"AtomicNumberTable: {tuple(s for s in self.zs)}"

    def index_to_z(self, index: int) -> int:
        return self.zs[index]

    def z_to_index(self, atomic_number: int) -> int:
        return self.zs.index(atomic_number)


def atomic_numbers_to_indices(z_table: AtomicNumberTable, atomic_numbers) -> torch.Tensor:
    """tools/atomic_number_table.py:37-43."""
    return torch.tensor([z_table.z_to_index(int(z)) for z in np.asarray(atomic_numbers).reshape(-1)], dtype=torch.long)


def atomic_symbols_to_indices(z_table: AtomicNumberTable, atomic_symbols) -> torch.Tensor:
    """tools/atomic_number_table.py:84-89."""
    return atomic_numbers_to_indices(z_table, [ATOMIC_NUMBER[s] for s in atomic_symbols])
