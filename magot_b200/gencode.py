"""NCBI genetic codes: the one place their tables live.

`codon64(n)` is the 64-byte table the C ABI takes (mg_plan_set_codon_table, mg_sixframe_count_table,
mg_translate_ascii_table): byte 16*b0 + 4*b1 + b2 (A=0 C=1 G=2 T=3) is the residue of codon b0 b1 b2, '*' a stop.
`library(n)` is the same code as a reference-style codon dict, for Sequence.translate(library=...).
`start64(codons, n)` is the 64-byte start-codon flag table mg_orfcall_count takes.

Tables 27, 28 and 31 read TAA/TAG/TGA as stop or sense depending on context, which a codon table cannot
express; they, 32 and the unassigned ids are refused.
"""

#: codon order of the NCBI strings: TTT TTC TTA TTG TCT ... (bases in TCAG order)
_TCAG = "TCAG"

#: id -> the 64 residues in NCBI (TCAG) codon order
TABLES = {
    1: "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    2: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNKKSS**VVVVAAAADDEEGGGG",
    3: "FFLLSSSSYY**CCWWTTTTPPPPHHQQRRRRIIMMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    4: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    5: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNKKSSSSVVVVAAAADDEEGGGG",
    6: "FFLLSSSSYYQQCC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    9: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIIMTTTTNNNKSSSSVVVVAAAADDEEGGGG",
    10: "FFLLSSSSYY**CCCWLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    11: "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    12: "FFLLSSSSYY**CC*WLLLSPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    13: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNKKSSGGVVVVAAAADDEEGGGG",
    14: "FFLLSSSSYYY*CCWWLLLLPPPPHHQQRRRRIIIMTTTTNNNKSSSSVVVVAAAADDEEGGGG",
    16: "FFLLSSSSYY*LCC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    21: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNNKSSSSVVVVAAAADDEEGGGG",
    22: "FFLLSS*SYY*LCC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    23: "FF*LSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    24: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSSKVVVVAAAADDEEGGGG",
    25: "FFLLSSSSYY**CCGWLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    26: "FFLLSSSSYY**CC*WLLLAPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    29: "FFLLSSSSYYYYCC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    30: "FFLLSSSSYYEECC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    33: "FFLLSSSSYYY*CCWWLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSSKVVVVAAAADDEEGGGG",
}

#: the supported ids, ascending
SUPPORTED = tuple(sorted(TABLES))


def check(genetic_code):
    """The id as an int; ValueError for anything that is not a supported NCBI table (strings from the command line
    included)."""
    try:
        n = int(genetic_code)
    except (TypeError, ValueError):
        n = None
    if n is None or isinstance(genetic_code, bool) or n not in TABLES or str(genetic_code).strip() != str(n):
        raise ValueError("genetic_code %r is not supported; supported NCBI tables: %s"
                         % (genetic_code, ", ".join(str(i) for i in SUPPORTED)))
    return n


def library(genetic_code):
    """Codon dict of the code in the reference's form (upper-case DNA codon -> one-letter residue, '*' = stop)."""
    t = TABLES[check(genetic_code)]
    return {_TCAG[i >> 4] + _TCAG[(i >> 2) & 3] + _TCAG[i & 3]: a for i, a in enumerate(t)}


def codon64(genetic_code):
    """The code as the C ABI's 64-byte table: byte 16*b0 + 4*b1 + b2, bases A=0 C=1 G=2 T=3."""
    lib = library(genetic_code)
    return bytes(ord(lib["ACGT"[i >> 4] + "ACGT"[(i >> 2) & 3] + "ACGT"[i & 3]]) for i in range(64))


def stops(genetic_code):
    """The code's stop codons, sorted."""
    return sorted(c for c, a in library(genetic_code).items() if a == "*")


def start64(codons, genetic_code=1):
    """Start codons (e.g. ("ATG", "GTG")) as the C ABI's 64 flags, byte 16*b0 + 4*b1 + b2 (A=0 C=1 G=2 T=3) = 1 for a start.
    ValueError for an empty list, a codon that is not three letters of A/C/G/T (either case) or a stop of the code."""
    code = check(genetic_code)
    if isinstance(codons, str):
        codons = [codons]
    codons = list(codons)
    if not codons:
        raise ValueError("no start codon given")
    lib = library(code)
    flags = bytearray(64)
    for c in codons:
        u = str(c).upper()
        if len(u) != 3 or any(b not in "ACGT" for b in u):
            raise ValueError("start codon %r is not three letters of A/C/G/T" % (c,))
        if lib[u] == "*":
            raise ValueError("start codon %s is a stop codon of genetic code %d" % (u, code))
        flags["ACGT".index(u[0]) * 16 + "ACGT".index(u[1]) * 4 + "ACGT".index(u[2])] = 1
    return bytes(flags)
