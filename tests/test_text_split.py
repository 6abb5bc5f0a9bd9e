"""Long-form text splitter (tortoise_tts_b200/text.py) against the reference's own known-answer tests and committed
outputs of the reference function on seeded synthetic texts."""
import importlib.util
import json
import os
import random

from tortoise_tts_b200.text import split_and_recombine_text, utterance_plan

HERE = os.path.dirname(os.path.abspath(__file__))


def test_reference_known_answers():
    """The two self-contained known-answer tests of the reference (utils/text.py:79-103)."""
    text = """
            This is a sample sentence.
            This is another sample sentence.
            This is a longer sample sentence that should force a split inthemiddlebutinotinthislongword.
            "Don't split my quote... please"
            """
    assert split_and_recombine_text(text, desired_length=20, max_length=40) == [
        'This is a sample sentence.',
        'This is another sample sentence.',
        'This is a longer sample sentence that',
        'should force a split',
        'inthemiddlebutinotinthislongword.',
        '"Don\'t split my quote... please"']
    text = """
            When you are really angry sometimes you use consecutive exclamation marks!!!!!! Is this a good thing to do?!?!?!
            I don't know but we should handle this situation..........................
            """
    assert split_and_recombine_text(text, desired_length=30, max_length=50) == [
        'When you are really angry sometimes you use',
        'consecutive exclamation marks!!!!!!',
        'Is this a good thing to do?!?!?!',
        'I don\'t know but we should handle this situation.']


def test_golden_vectors():
    with open(os.path.join(HERE, "golden", "text_split_v1.json")) as f:
        cases = json.load(f)
    assert len(cases) >= 40
    for c in cases:
        assert split_and_recombine_text(c["text"], c["desired_length"], c["max_length"]) == c["chunks"], c["text"][:80]


def test_properties():
    """No chunk is empty or punctuation-only, none exceeds max_length, and no non-space character is lost or reordered."""
    rng = random.Random(7)
    for _ in range(50):
        words = ["w%d" % rng.randint(0, 999) + rng.choice(["", ".", "!", "?", ","]) for _ in range(rng.randint(1, 300))]
        text = " ".join(words)
        d = rng.choice([20, 50, 200])
        m = d + rng.choice([10, 100])
        chunks = split_and_recombine_text(text, d, m)
        assert all(0 < len(c) <= m for c in chunks)
        assert "".join("".join(chunks).split()) == "".join(text.split())


def test_utterance_plan():
    assert utterance_plan(5, 1) == [0, 0, 0, 0, 0]
    assert utterance_plan(5, 2) == [0, 1, 0, 1, 0]
    assert utterance_plan(3, 8) == [0, 1, 2]


def test_against_reference_function():
    """Digests of the reference function's chunks on seeded random texts and on its own sample story are stored
    (tests/ref_golden.py); the story itself is stored with them."""
    import ref_golden as rg

    def reference_module():
        from oracle.ref_shims import REFERENCE_ROOT
        spec = importlib.util.spec_from_file_location("ref_text", os.path.join(REFERENCE_ROOT, "tortoise", "utils", "text.py"))
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
        return ref
    rng = random.Random(99)
    alphabet = 'abc de. fg! "hi?" \n\n jk... “lm” ,;:x' + "y" * 5
    for i in range(400):
        text = "".join(rng.choice(alphabet) for _ in range(rng.randint(0, 500)))
        d = rng.choice([5, 20, 60, 200])
        m = d + rng.choice([1, 10, 100])
        want = rg.digest("text_split_%d" % i, lambda: reference_module().split_and_recombine_text(text, d, m))
        assert rg.hexdigest(split_and_recombine_text(text, d, m)) == want, repr(text)

    def reference_story():
        from oracle.ref_shims import REFERENCE_ROOT
        with open(os.path.join(REFERENCE_ROOT, "tortoise", "data", "riding_hood.txt")) as f:
            return f.read()
    t = rg.value("text_split_story", reference_story)
    want = rg.digest("text_split_story_chunks", lambda: reference_module().split_and_recombine_text(t))
    assert rg.hexdigest(split_and_recombine_text(t)) == want
