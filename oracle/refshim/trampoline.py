"""Minimal stand-in for the pure-Python `trampoline` package (setup.py:46 of the reference), which
torch does not depend on and may not be installed.  Used only to import the reference: by the golden
generators under tests/golden/ and next to the copy that oracle/stage_reference.py stages; semantics per its usage in torchsde/_brownian/brownian_interval.py:183-315:
run a generator; a yielded generator is run and its return value sent back; `raise TailCall(g)`
replaces the current frame by g."""
class TailCall(Exception):
    def __init__(self, gen): self.gen = gen
def trampoline(gen):
    stack = [gen]; send = None
    while stack:
        g = stack[-1]
        try:
            y = g.send(send); send = None
            stack.append(y)
        except StopIteration as e:
            stack.pop(); send = e.value
        except TailCall as e:
            stack.pop(); stack.append(e.gen); send = None
    return send
