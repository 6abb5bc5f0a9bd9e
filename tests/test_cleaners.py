"""CPU: the tokenizer's text cleaners (tortoise_tts_b200/cleaners.py) against the known-answer table of the upstream
cleaners the reference vendors (tortoise/utils/tokenizer.py:11-157 is keithito/tacotron `text/cleaners.py` + `numbers.py`;
the expectations below are that project's published unit-test vectors for normalize_numbers, which the reference does
not ship) and against the reference's own `english_cleaners` on number-free text (`inflect` is absent from this image,
so the reference cannot expand numbers here)."""
import pytest

from tortoise_tts_b200 import cleaners as c

NUMBERS = [
    ("1", "one"), ("15", "fifteen"), ("24", "twenty-four"), ("100", "one hundred"), ("101", "one hundred one"),
    ("456", "four hundred fifty-six"), ("1000", "one thousand"), ("1800", "eighteen hundred"), ("2,000", "two thousand"),
    ("3000", "three thousand"), ("18000", "eighteen thousand"), ("24,000", "twenty-four thousand"),
    ("124,001", "one hundred twenty-four thousand one"), ("6.4 sec", "six point four sec"),
    ("1st", "first"), ("2nd", "second"), ("9th", "ninth"), ("243rd place", "two hundred and forty-third place"),
    ("1400", "fourteen hundred"), ("1901", "nineteen oh one"), ("1999", "nineteen ninety-nine"), ("2000", "two thousand"),
    ("2004", "two thousand four"), ("2010", "twenty ten"), ("2012", "twenty twelve"), ("2025", "twenty twenty-five"),
    ("September 11, 2001", "September eleven, two thousand one"),
    ("July 26, 1984.", "July twenty-six, nineteen eighty-four."),
    ("$0.00", "zero dollars"), ("$1", "one dollar"), ("$10", "ten dollars"), ("$.01", "one cent"),
    ("$0.25", "twenty-five cents"), ("$5.00", "five dollars"), ("$5.01", "five dollars, one cent"),
    ("$135.99.", "one hundred thirty-five dollars, ninety-nine cents."), ("$40,000", "forty thousand dollars"),
    ("for £2500!", "for twenty-five hundred pounds!"),
    ("0", "zero"), ("1234567", "one million, two hundred thirty-four thousand, five hundred sixty-seven"),
    ("12th", "twelfth"), ("20th", "twentieth"), ("100th", "one hundredth"), ("21st", "twenty-first"),
]


@pytest.mark.parametrize("src,want", NUMBERS)
def test_normalize_numbers(src, want):
    assert c.normalize_numbers(src) == want


def test_english_cleaners_chain():
    assert c.english_cleaners('Mr. Smith paid  $5.01 to Dr. "Who" on the 3rd.') == \
        "mister smith paid five dollars, one cent to doctor who on the third."
    assert c.english_cleaners("St. John's Ft. Knox, Ltd.") == "saint john's fort knox, limited"
    assert c.basic_cleaners('A  "B"\n c') == 'a "b" c'           # basic cleaners keep quotes (tokenizer.py:129-133)
    assert c.english_cleaners("naïve café – “déjà vu”…") == "naive cafe - deja vu..."
    assert c.to_ascii("plain ascii 123") == "plain ascii 123"


def test_against_reference_cleaners_without_numbers():
    """Digests of the reference's english_cleaners / basic_cleaners outputs are stored (tests/ref_golden.py)."""
    import random
    import ref_golden as rg
    rng = random.Random(0)
    words = ["Mr.", "Mrs.", "Dr.", "St.", "the", "Quick", "BROWN", "fox,", '"quoted"', "co.", "Ltd.", "hello\tworld",
             "Gen.", "lt.", "end.", "  spaced  ", "semi;colon", "Capt.", "jr.", "x"]

    def reference(s):
        from oracle import ref_shims
        ref_shims.load_reference()
        from tortoise.utils import tokenizer as rt
        return [rt.english_cleaners(s), rt.basic_cleaners(s)]
    for i in range(200):
        s = " ".join(rng.choice(words) for _ in range(rng.randint(1, 12)))
        assert rg.hexdigest([c.english_cleaners(s), c.basic_cleaners(s)]) == \
            rg.digest("cleaners_%d" % i, lambda: reference(s)), s
