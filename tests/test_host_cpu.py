"""CPU tests of the product's host side (C++ mirror of the reference's llmclient + Task LLM step,
chat template, tokenizer, tool-call extraction) against the oracle and the reference's goldens.
No GPU: only JSON-in/JSON-out hooks of include/acp_host.h are called."""
import copy
import json
import os
import re

import pytest

from agentcontrolplane_b200 import host
from oracle import boundary as B
from oracle import chat_oracle as C

G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_goldens.json")))
FX = G["fixtures"]

TOOLS_WIRE = [{"type": "function", "function": {"name": "fetch__fetch", "description": "Fetch a URL",
                                                 "parameters": {"type": "object", "properties": {"url": {"type": "string"}}, "required": ["url"]}}}]


def _task(phase="ReadyForLLM", window=None, name=None):
    return {"metadata": {"name": name or FX["task_name"], "namespace": "default", "uid": "uid-1"},
            "spec": {"agentRef": {"name": FX["agent_name"]}},
            "status": {"phase": phase, "status": "Ready", "contextWindow": window if window is not None else [
                {"role": "system", "content": FX["system_prompt"]}, {"role": "user", "content": FX["user_message"]}]}}


def _reasons(out):
    return [e["reason"] for e in out["events"]]


def _oracle_step(task, tools, mock):
    class Cl:
        def send_request(self, messages, tools):
            if "error" in mock:
                raise RuntimeError(mock["error"])
            if "request_error" in mock:
                raise B.LLMRequestError(mock["request_error"]["status"], mock["request_error"]["message"])
            return copy.deepcopy(mock["message"])
    t, rec, tcs = copy.deepcopy(task), B.Recorder(), []
    res, err = B.send_llm_request(t, tools, Cl(), rec, tcs)
    return t, res, err, rec, tcs


# ------------------------------------------------------------------ Task step: goldens + oracle
def test_G1_final_answer_host_matches_reference_and_oracle():
    g = G["G1_final_answer"]
    out = host.task_step({"op": "sendLLMRequest", "task": _task(), "tools": [],
                          "llm": {"provider": "mock", "mock": {"message": g["llm_output"]}}})
    st = out["task"]["status"]
    assert st["phase"] == "FinalAnswer" and "LLM final response received" in st["statusDetail"]
    assert st["output"] == g["llm_output"]["content"]
    assert len(st["contextWindow"]) == 3 and st["contextWindow"][2]["role"] == "assistant"
    assert out["result"] == {"requeue": False, "requeueAfter": 0} and out["error"] == ""
    assert "SendingContextWindowToLLM" in _reasons(out) and "LLMFinalAnswer" in _reasons(out)
    ot, _, _, orec, _ = _oracle_step(_task(), [], {"message": g["llm_output"]})
    for k in ("phase", "output", "statusDetail", "status"):
        assert st[k] == ot["status"][k]
    assert st["contextWindow"] == ot["status"]["contextWindow"]
    assert _reasons(out) == [r for (_, r, _) in orec.events]
    # API traffic of the reference: lease create, status write, final status write, lease delete
    assert out["store_writes"] == 4


def test_G2_tool_call_host():
    g = G["G2_tool_call"]
    tools = B.convert_mcp_tools([{"name": "fetch", "description": "d"}], "fetch")
    out = host.task_step({"op": "sendLLMRequest", "task": _task(window=[]), "tools": tools,
                          "llm": {"provider": "mock", "mock": {"message": g["llm_output"]}}})
    st = out["task"]["status"]
    assert st["phase"] == "ToolCallsPending" and out["result"]["requeueAfter"] == 5
    assert len(out["toolcalls"]) == 1
    tc = out["toolcalls"][0]
    assert tc["spec"]["toolRef"]["name"] == "fetch__fetch"
    assert tc["spec"]["arguments"] == g["expect"]["arguments"]            # byte-identical
    assert tc["spec"]["toolType"] == "MCP" and tc["spec"]["toolCallId"] == "1"
    rid = st["toolCallRequestId"]
    assert re.match(G["G10_id_format"]["regex"], rid) and len(rid) == 7
    assert tc["metadata"]["name"] == "%s-%s-tc-%02d" % (FX["task_name"], rid, 1)
    assert tc["metadata"]["labels"] == {"acp.humanlayer.dev/task": FX["task_name"], "acp.humanlayer.dev/toolcallrequest": rid}
    assert tc["metadata"]["ownerReferences"][0]["controller"] is True
    assert "ToolCallsPending" in _reasons(out) and "ToolCallCreated" in _reasons(out)


def test_G3_G4_errors_host():
    g3 = G["G3_generic_error"]
    out = host.task_step({"op": "sendLLMRequest", "task": _task(), "tools": [],
                          "llm": {"provider": "mock", "mock": {"error": g3["error"]}}})
    st = out["task"]["status"]
    assert out["error"] == g3["error"] and out["result"]["requeueAfter"] == 5
    assert st["status"] == "Error" and st["phase"] == "ReadyForLLM" and st["error"] == g3["error"]
    assert "LLMRequestFailed" in _reasons(out)
    g4 = G["G4_4xx_error"]
    out = host.task_step({"op": "sendLLMRequest", "task": _task(), "tools": [],
                          "llm": {"provider": "mock", "mock": {"request_error": {"status": g4["status_code"], "message": g4["message"]}}}})
    st = out["task"]["status"]
    assert out["error"] == "" and out["result"] == {"requeue": False, "requeueAfter": 0}
    assert st["status"] == "Error" and st["phase"] == "Failed"
    assert g4["expect"]["error_contains"] in st["error"] and "LLMRequestFailed4xx" in _reasons(out)
    ot, _, _, _, _ = _oracle_step(_task(), [], {"request_error": {"status": 400, "message": g4["message"]}})
    assert st["error"] == ot["status"]["error"] and st["statusDetail"] == ot["status"]["statusDetail"]


def test_G5_check_tool_calls_host():
    g = G["G5_tool_results_fold_back"]
    window = [{"role": "system", "content": FX["system_prompt"]}, {"role": "user", "content": FX["user_message"]},
              {"role": "assistant", "content": "", "toolCalls": [
                  {"id": "1", "type": "function", "function": {"name": "fetch__fetch", "arguments": "{}"}},
                  {"id": "2", "type": "function", "function": {"name": "fetch__fetch", "arguments": "{}"}}]}]
    task = _task(phase="ToolCallsPending", window=window)
    task["status"]["toolCallRequestId"] = "abc1234"

    def tcs(statuses):
        return [{"metadata": {"name": f"{FX['task_name']}-abc1234-tc-{i + 1:02d}", "namespace": "default",
                              "labels": {"acp.humanlayer.dev/task": FX["task_name"], "acp.humanlayer.dev/toolcallrequest": "abc1234"}},
                 "spec": {"toolCallId": t["spec"]["toolCallId"], "taskRef": {"name": FX["task_name"]},
                          "toolRef": {"name": "fetch__fetch"}, "toolType": "MCP", "arguments": "{}"},
                 "status": {"status": s, "result": t["status"]["result"]}} for i, (t, s) in enumerate(zip(g["toolcalls"], statuses))]
    out = host.task_step({"op": "checkToolCalls", "task": task, "toolcalls": tcs(["Succeeded", "Running"])})
    assert out["result"]["requeueAfter"] == 5 and out["task"]["status"]["phase"] == "ToolCallsPending"
    out = host.task_step({"op": "checkToolCalls", "task": task, "toolcalls": tcs(["Succeeded", "Error"])})
    st = out["task"]["status"]
    assert out["result"]["requeue"] is True and st["phase"] == "ReadyForLLM" and len(st["contextWindow"]) == 5
    for t, m in zip(g["toolcalls"], st["contextWindow"][3:]):
        assert m == {"role": "tool", "content": t["status"]["result"], "toolCallId": t["spec"]["toolCallId"]}


def test_unsupported_provider_fails_like_the_reference():
    out = host.task_step({"op": "sendLLMRequest", "task": _task(), "tools": [], "llm": {"provider": "bogus"}})
    st = out["task"]["status"]
    assert st["phase"] == "Failed" and "unsupported provider: bogus" in st["error"]
    assert "LLMClientCreationFailed" in _reasons(out)
    out = host.task_step({"op": "sendLLMRequest", "task": _task(), "tools": [], "llm": {"provider": "local"}})
    assert out["task"]["status"]["phase"] == "Failed"      # no engine in this process: loud, no fallback


# ------------------------------------------------------------------ wire conversion
def test_request_body_matches_oracle():
    window = [{"role": "system", "content": "s"}, {"role": "user", "content": "u \"q\" é"},
              {"role": "assistant", "content": "", "toolCalls": [{"id": "1", "type": "function", "function": {"name": "f__g", "arguments": "{\"a\": 1}"}}]},
              {"role": "tool", "content": "42", "toolCallId": "1"}, {"role": "weird", "content": "w"}]
    tools = B.convert_mcp_tools([{"name": "g", "description": "d", "inputSchema": {"type": "object", "properties": {"a": {"type": "number"}}}}], "f")
    got = host.build_chat_request("m", window, tools)
    want = B.build_chat_request("m", window, tools)
    assert got == want
    assert "acpToolType" not in json.dumps(got)
    assert "tools" not in host.build_chat_request("m", window, [])


def test_response_flattening_matches_reference_fixtures():
    g = G["G8_wire_fixtures"]
    assert host.convert_response(g["content_body"]["body"]) == {"role": "assistant", "content": "test"}
    m = host.convert_response(g["tool_body"]["body"])
    e = g["tool_body"]["expect_tool"]
    assert m["content"] == "" and m["toolCalls"] == [{"id": e["id"], "function": {"name": e["name"], "arguments": e["arguments"]}, "type": e["type"]}]
    both = {"choices": [{"message": {"content": "hi"}}, {"message": {"content": "x", "tool_calls": [{"id": "a", "type": "function", "function": {"name": "n", "arguments": "{}"}}]}}]}
    assert host.convert_response(both) == {k: v for k, v in B.convert_from_response(both).items()} | {"toolCalls": [{"id": "a", "function": {"name": "n", "arguments": "{}"}, "type": "function"}]}
    assert host.convert_response({"choices": []}) == {"role": "assistant", "content": ""}


# ------------------------------------------------------------------ template / tokenizer / parser
CASES = [
    ([{"role": "system", "content": "You are a helpful test assistant."}, {"role": "user", "content": "What is the capital of France?"}], []),
    ([{"role": "user", "content": "no system"}], []),
    ([{"role": "system", "content": "sys"}, {"role": "user", "content": "use a tool ☃"},
      {"role": "assistant", "content": None, "tool_calls": [{"id": "c1", "type": "function", "function": {"name": "fetch__fetch", "arguments": "{\"url\": \"https://api.example.com/data\"}"}}]},
      {"role": "tool", "tool_call_id": "c1", "content": "{\"data\": \"test-data\"}"}], TOOLS_WIRE),
    ([{"role": "user", "content": "a"}, {"role": "assistant", "content": "b"}, {"role": "system", "content": "mid"}, {"role": "odd", "content": "c"}], TOOLS_WIRE),
]


@pytest.mark.parametrize("messages,tools", CASES)
def test_template_matches_oracle(messages, tools):
    req = {"messages": messages}
    if tools:
        req["tools"] = tools
    got = host.render_prompt(req)
    ids, text = C.render(messages, tools)
    assert got["text"] == text
    assert got["token_ids"] == ids
    assert ids[0] == 128000 and ids[-3:] == [128007, 10, 10]
    # byte-level tokenizer: every non-special id is the UTF-8 byte
    assert bytes(t for t in ids if t < 256).decode() == re.sub(r"<\|[a-z_]+\|>", "", text)


def test_request_validation_statuses():
    assert host.render_prompt({"messages": []})["status"] == 400
    assert host.render_prompt({"messages": [{"content": "x"}]})["status"] == 400
    assert host.render_prompt({"messages": [{"role": "user", "content": "x"}], "stream": True})["status"] == 400
    assert host.render_prompt({"messages": [{"role": "user", "content": "x"}], "max_tokens": 0})["status"] == 400
    assert host.render_prompt({"messages": [{"role": "user", "content": "x"}], "temperature": -1})["status"] == 400
    r = host.render_prompt({"messages": [{"role": "user", "content": [{"type": "text", "text": "parts"}]}]})
    assert "parts" in r["text"]


def test_decode_tokens_matches_oracle():
    ids = list(range(0, 300)) + [1000, 65791, 65792, 127999, 128000, 128009, 128255, 33709, 42410]
    assert host.decode_tokens(ids) == C.decode_tokens(ids)
    assert host.decode_tokens([72, 105]) == b"Hi"


PARSE_CASES = [
    '{"name": "fetch__fetch", "parameters": {"url": "https://api.example.com/data"}}',
    '  {"name":"fetch__fetch","parameters":{"url":  "x", "n": [1, 2, {"a": "}"}]}}\n',
    '{"name": "fetch__fetch", "parameters": {"url": "a"}}\n{"name": "fetch__fetch", "parameters": {"url": "b"}}',
    '{"name": "unknown_tool", "parameters": {}}',
    '{"name": "fetch__fetch", "parameters": "not an object"}',
    'The answer is {"name": "fetch__fetch"}',
    '{"name": "fetch__fetch", "parameters": {"url": "a"}} trailing words',
    'plain final answer', '', '{"broken": ',
    '{"name": "fetch__fetch", "arguments": {"url": "\\u00e9\\n"}}',
]


@pytest.mark.parametrize("text", PARSE_CASES)
def test_parse_completion_matches_oracle(text):
    got = host.parse_completion(text, TOOLS_WIRE, "call_7_")
    want = C.parse_completion(text, TOOLS_WIRE, "call_7_")
    assert got == want
    if "tool_calls" in got:
        for tc in got["tool_calls"]:
            assert tc["function"]["arguments"] in text            # verbatim substring
            assert isinstance(json.loads(tc["function"]["arguments"]), dict)
    assert host.parse_completion(text, [], "c") == {"content": text}   # no tools -> always content


# ------------------------------------------------------------------ CPU reconcile loop over the stub server
def test_config0_plumbing_over_stub_server():
    """BASELINE config 0: 1 Task, stub completion server returning the reference's fixture body,
    the reference's own (restated) openai path — no GPU anywhere."""
    with host.StubServer() as srv:
        out = host.task_step({"op": "sendLLMRequest", "task": _task(window=[
            {"role": "system", "content": G["G8_wire_fixtures"]["window"]["system"]},
            {"role": "user", "content": G["G8_wire_fixtures"]["window"]["user"]}]), "tools": [],
            "llm": {"provider": "openai", "model": "gpt-4o", "baseURL": srv.base_url}})
        st = out["task"]["status"]
        assert st["phase"] == "FinalAnswer" and st["output"] == "test" and len(st["contextWindow"]) == 3
        r = host.hostsim_run({"tasks": 200, "workers": 4, "provider": "openai", "model": "gpt-4o", "baseURL": srv.base_url})
        assert r["reconciles"] == 200 and r["final_phases"] == {"FinalAnswer": 200}
        assert r["store_writes"] >= 4 * 200 and r["reconciles_per_s"] > 0 and "outputs" not in r
        r = host.hostsim_run({"tasks": 20, "workers": 4, "provider": "openai", "model": "gpt-4o", "baseURL": srv.base_url,
                              "return_outputs": True})
        assert r["outputs"] == ["test"] * 20
    tool_body = G["G8_wire_fixtures"]["tool_body"]["body"]
    with host.StubServer(tool_body) as srv:
        out = host.task_step({"op": "sendLLMRequest", "task": _task(), "tools": B.convert_mcp_tools([{"name": "fetch"}], "fetch"),
                              "llm": {"provider": "openai", "model": "gpt-4o", "baseURL": srv.base_url}})
        assert out["task"]["status"]["phase"] == "ToolCallsPending"
        assert out["toolcalls"][0]["spec"]["arguments"] == G["G8_wire_fixtures"]["tool_body"]["expect_tool"]["arguments"]
        assert out["toolcalls"][0]["spec"]["toolCallId"] == "tool-call-1"


def test_connection_refused_is_a_retryable_error():
    out = host.task_step({"op": "sendLLMRequest", "task": _task(), "tools": [],
                          "llm": {"provider": "openai", "model": "m", "baseURL": "http://127.0.0.1:9/v1"}})
    assert out["error"].startswith("model API call failed") and out["task"]["status"]["phase"] == "ReadyForLLM"


def test_hostsim_window_sizing_reports_real_length():
    """The synthetic window hits its token target exactly; when the agent's tool schemas alone exceed
    it (byte-level synthetic tokenizer) the reported length is the real one, never a failure."""
    assert host.hostsim_window_tokens(512, 0) == 512
    assert host.hostsim_window_tokens(1024, 2) == 1024
    small = host.hostsim_window_tokens(64, 2)
    assert small > 64 and small == host.hostsim_window_tokens(1, 2)


def test_unimplemented_completion_parameters_are_refused_not_ignored():
    """stop / tool_choice / logprobs / response_format would change the completion: a request that sets
    them gets a 400 (terminal LLMRequestError upstream) instead of a silently different answer; their
    neutral spellings pass."""
    base = {"model": "m", "messages": [{"role": "user", "content": "hi"}]}
    for extra in ({}, {"stop": []}, {"stop": None}, {"tool_choice": "auto"}, {"logprobs": False}, {"response_format": {"type": "text"}}):
        assert "status" not in host.render_prompt(dict(base, **extra)), extra
    for extra, needle in (({"stop": ["\n"]}, "stop"), ({"stop": "x"}, "stop"), ({"tool_choice": "required"}, "tool_choice"),
                          ({"tool_choice": {"type": "function", "function": {"name": "f"}}}, "tool_choice"),
                          ({"logprobs": True}, "logprobs"), ({"response_format": {"type": "json_object"}}, "response_format"),
                          ({"frequency_penalty": 0.5}, "frequency_penalty"), ({"presence_penalty": -1}, "presence_penalty")):
        r = host.render_prompt(dict(base, **extra))
        assert r.get("status") == 400 and needle in r["error"], (extra, r)


# ------------------------------------------------------------------ a5 / a6 / a8: the cluster lookups of the LLM step
def _agent(ready=True, **spec):
    return {"metadata": {"name": FX["agent_name"], "namespace": "default"},
            "spec": dict({"llmRef": {"name": "test-llm"}, "system": FX["system_prompt"]}, **spec),
            "status": {"ready": ready, "validHumanContactChannels": spec.pop("_channels", [])}}


def _llm(provider="mock", key_from=True, **params):
    spec = {"provider": provider, "parameters": dict({"model": "m"}, **params)}
    if key_from:
        spec["apiKeyFrom"] = {"secretKeyRef": {"name": "test-secret", "key": "api-key"}}
    return {"metadata": {"name": "test-llm"}, "spec": spec}


SECRET = {"metadata": {"name": "test-secret"}, "data": {"api-key": "sk-test"}}


def _cluster_step(objects, mcp=None, task=None):
    return host.task_step({"op": "sendLLMRequestFromCluster", "task": task or _task(), "mcp": mcp or {},
                           "objects": [{"kind": k, "object": o} for k, o in objects]})


def test_G12_G13_validate_task_and_agent_host_matches_reference_and_oracle():
    for gname, objects, agent in (("G12_agent_missing", [], None),
                                  ("G13_agent_not_ready", [("Agent", _agent(ready=False))], _agent(ready=False))):
        exp = G[gname]["expect"]
        out = _cluster_step(objects)
        st = out["task"]["status"]
        assert st["phase"] == exp["phase"] and st["status"] == exp["status"]
        assert exp["statusDetail_contains"] in st["statusDetail"] and st.get("error", "") == ""
        assert out["result"]["requeueAfter"] == exp["requeue_after"] and out["error"] == ""
        for frag in exp["events_containing"]:
            assert any(frag in e["reason"] or frag in e["message"] for e in out["events"])
        ot, rec = _task(), B.Recorder()
        res = B.validate_task_and_agent(ot, agent, rec)
        assert res.requeue_after == exp["requeue_after"]
        for k in ("phase", "status", "statusDetail"):
            assert st[k] == ot["status"][k]
        assert [(e["type"], e["reason"], e["message"]) for e in out["events"]] == rec.events


def test_get_llm_and_credentials_failures_match_oracle():
    cases = [
        ([("Agent", _agent())], None, {}, "LLMFetchFailed"),
        ([("Agent", _agent()), ("LLM", _llm("openai"))], _llm("openai"), {}, "APIKeySecretFetchFailed"),
        ([("Agent", _agent()), ("LLM", _llm("openai")), ("Secret", {"metadata": {"name": "test-secret"}, "data": {"api-key": ""}})],
         _llm("openai"), {"test-secret": {"data": {"api-key": ""}}}, "EmptyAPIKey"),
    ]
    for objects, llm, secrets_by_name, reason in cases:
        out = _cluster_step(objects)
        st = out["task"]["status"]
        ot, rec = _task(), B.Recorder()
        key, err = B.get_llm_and_credentials(ot, llm, "test-llm", secrets_by_name, rec)
        assert key is None and err
        assert st["phase"] == "Failed" and st["status"] == "Error"
        assert st["error"] == ot["status"]["error"] == err == out["error"]
        assert st["statusDetail"] == ot["status"]["statusDetail"]
        assert _reasons(out) == [reason] == [r for (_, r, _) in rec.events]
        assert out["result"] == {"requeue": False, "requeueAfter": 0}


def test_local_provider_needs_no_secret_and_other_providers_do():
    """INTEGRATION.md §4: with provider `local` and no apiKeyFrom the reference would dereference a nil
    pointer (state_machine.go:504); the mirror skips the Secret and goes on to CreateClient — which,
    without an engine in this CPU test, fails with the typed client-creation error, proving the
    credentials step was passed."""
    out = _cluster_step([("Agent", _agent()), ("LLM", _llm("local", key_from=False))])
    st = out["task"]["status"]
    assert _reasons(out) == ["LLMClientCreationFailed"]
    assert st["phase"] == "Failed" and "engine not initialised" in st["error"]
    ot, rec = _task(), B.Recorder()
    assert B.get_llm_and_credentials(ot, _llm("local", key_from=False), "test-llm", {}, rec) == ("", None)
    # an unknown provider with valid credentials reaches the provider switch (langchaingo_client.go:71-72)
    out = _cluster_step([("Agent", _agent()), ("LLM", _llm("cohere")), ("Secret", SECRET)])
    assert "unsupported provider: cohere" in out["task"]["status"]["error"]


def test_G14_contact_channel_tools_and_collect_tools_order():
    g = G["G14_contact_channel_tools"]
    for case in g["cases"]:
        agent = _agent()
        agent["status"]["validHumanContactChannels"] = [{"name": case["channel"]["metadata"]["name"]}]
        out = host.task_step({"op": "collectTools", "task": _task(), "agent": agent, "mcp": {},
                              "objects": [{"kind": "ContactChannel", "object": case["channel"]}]})
        (tool,) = out["tools"]
        assert tool["function"]["name"] == case["name"] and tool["function"]["description"] == case["description"]
        assert tool["function"]["parameters"] == g["parameters"] and tool["acpToolType"] == g["acpToolType"]
        assert tool == B.tool_from_contact_channel({"name": case["channel"]["metadata"]["name"], "spec": case["channel"]["spec"]})
    # order: MCP servers (agent order, unknown servers skipped), contact channels, sub-agents (missing ones skipped)
    agent = _agent(mcpServers=[{"name": "fetch"}, {"name": "ghost"}, {"name": "files"}], subAgents=[{"name": "sub-agent"}, {"name": "gone"}])
    agent["status"]["validHumanContactChannels"] = [{"name": "ops"}]
    mcp = {"files": [{"name": "read", "description": "Read a file", "inputSchema": {"type": "object", "properties": {"path": {"type": "string"}}}}],
           "fetch": [{"name": "fetch", "description": "Fetch a URL"}]}
    channel = G["G14_contact_channel_tools"]["cases"][0]["channel"]
    sub = {"metadata": {"name": "sub-agent"}, "spec": {"description": G["G7_delegate_tool"]["agent"]["description"]}}
    out = host.task_step({"op": "collectTools", "task": _task(), "agent": agent, "mcp": mcp,
                          "objects": [{"kind": "ContactChannel", "object": channel}, {"kind": "Agent", "object": sub}]})
    names = [t["function"]["name"] for t in out["tools"]]
    assert names == ["fetch__fetch", "files__read", "ops__human_contact_email", "delegate_to_agent__sub-agent"]
    want = B.collect_tools(agent, mcp, {"ops": channel}, {"sub-agent": sub})
    assert out["tools"] == want
    assert B.build_tool_type_map(want) == {"fetch__fetch": "MCP", "files__read": "MCP", "ops__human_contact_email": "HumanContact",
                                           "delegate_to_agent__sub-agent": "DelegateToAgent"}


def test_local_client_forwards_llm_parameters():
    """a20: temperature / topP / topK / maxTokens of LLM.spec.parameters (llm_types.go:41-71) reach the
    engine's request body; without them the body says temperature 0 like the reference's wire."""
    body = host.build_chat_request("m", [{"role": "user", "content": "hi"}], [])
    assert body["temperature"] == 0 and "top_p" not in body and "top_k" not in body and "max_tokens" not in body


# ------------------------------------------------------------------ a1 / a2 / a4: Reconcile, Process, lease, mutex
def _objs(*pairs):
    return [{"kind": k, "object": o} for k, o in pairs]


def test_process_walks_the_phases_of_the_reference_state_machine():
    """StateMachine.Process (state_machine.go:84-114) from an empty status to FinalAnswer, one Reconcile
    at a time, against the stub completion server (provider openai over loopback)."""
    with host.StubServer() as srv:
        llm = _llm("openai", baseUrl=srv.base_url)
        cluster = _objs(("Agent", _agent()), ("LLM", llm), ("Secret", SECRET))
        task = {"metadata": {"name": FX["task_name"], "namespace": "default", "uid": "uid-1"},
                "spec": {"agentRef": {"name": FX["agent_name"]}, "userMessage": FX["user_message"]}, "status": {}}
        # "" -> Initializing (initialize, :119-146)
        out = host.task_step({"op": "process", "task": task, "objects": cluster})
        st = out["task"]["status"]
        assert (st["phase"], st["status"], st["statusDetail"]) == ("Initializing", "Pending", "Initializing Task")
        assert out["result"] == {"requeue": True, "requeueAfter": 0}
        # Initializing -> ReadyForLLM (validateAgent + prepareForLLM, task_controller_test.go:306-341)
        out = host.task_step({"op": "process", "task": out["task"], "objects": cluster})
        st = out["task"]["status"]
        assert st["phase"] == "ReadyForLLM" and st["ready"] and "Ready to send to LLM" in st["statusDetail"]
        assert [m["role"] for m in st["contextWindow"]] == ["system", "user"]
        assert st["contextWindow"][0]["content"] == FX["system_prompt"] and st["contextWindow"][1]["content"] == FX["user_message"]
        assert _reasons(out) == ["ValidationSucceeded"] and out["result"]["requeue"] is True
        # ReadyForLLM -> FinalAnswer (sendLLMRequest; the stub answers G8's content body)
        out = host.task_step({"op": "process", "task": out["task"], "objects": cluster})
        st = out["task"]["status"]
        assert st["phase"] == "FinalAnswer" and st["output"] == G["G8_wire_fixtures"]["content_body"]["expect_content"]
        assert "lease" not in out                      # released (deleted) at the end of the step
        assert out["store_writes"] == 4                # lease create, "Sending request" status write, final status write, lease delete
        # terminal: nothing happens any more (handleTerminal)
        out2 = host.task_step({"op": "process", "task": out["task"], "objects": cluster})
        assert out2["task"]["status"] == out["task"]["status"] and out2["events"] == [] and out2["result"] == {"requeue": False, "requeueAfter": 0}


def test_prepare_for_llm_validation_errors_match_the_reference():
    ve = G["G6_initial_window"]["validation_errors"]
    window = [{"role": "user", "content": "hi"}]
    for spec, want in (({"userMessage": "x", "contextWindow": window}, ve["both"]), ({}, ve["neither"]),
                       ({"contextWindow": [{"role": "system", "content": "s"}]}, ve["no_user"])):
        task = {"metadata": {"name": FX["task_name"]}, "spec": dict({"agentRef": {"name": FX["agent_name"]}}, **spec),
                "status": {"phase": "Initializing", "status": "Pending"}}
        out = host.task_step({"op": "process", "task": task, "objects": _objs(("Agent", _agent()))})
        st = out["task"]["status"]
        assert st["phase"] == "Failed" and st["error"] == want == out["error"] and _reasons(out) == ["ValidationFailed"]
        assert B.validate_task_message_input(spec.get("userMessage", ""), spec.get("contextWindow", [])) == want


def test_reconcile_ignores_a_missing_task_and_dispatches_an_existing_one():
    out = host.task_step({"op": "reconcile", "name": "ghost", "task": _task(), "objects": []})
    assert out["result"] == {"requeue": False, "requeueAfter": 0} and out["error"] == "" and out["events"] == []
    t = _task(phase="Pending")
    out = host.task_step({"op": "reconcile", "name": FX["task_name"], "task": t, "objects": _objs(("Task", t))})
    assert out["task"]["status"]["statusDetail"] == "Waiting for Agent to exist" and out["result"]["requeueAfter"] == 5


def test_task_lease_follows_the_reference_rules():
    """acquireTaskLease / canAcquireLease (state_machine.go:1069-1132): a live lease of another pod
    defers the step by 5 s without touching the Task; an expired one (renewTime + 30 s) or our own is
    taken over; provider `local` may skip the lease altogether."""
    def lease(holder, renew):
        return {"metadata": {"name": "task-llm-" + FX["task_name"]}, "spec": {"holderIdentity": holder, "leaseDurationSeconds": 30,
                                                                             "acquireTime": renew, "renewTime": renew}}
    base = {"op": "sendLLMRequest", "task": _task(), "tools": [], "llm": {"provider": "mock", "mock": {"message": G["G1_final_answer"]["llm_output"]}}}
    cluster = _objs(("Agent", _agent()), ("LLM", _llm("cohere")), ("Secret", SECRET))
    # another pod renewed 10 s ago: held
    out = host.task_step({"op": "process", "task": _task(), "now": 1000.0, "podName": "pod-a",
                          "objects": cluster + _objs(("Lease", lease("pod-b", 990.0)))})
    assert out["result"] == {"requeue": False, "requeueAfter": 5} and out["events"] == []
    assert out["task"]["status"]["phase"] == "ReadyForLLM" and out["lease"]["spec"]["holderIdentity"] == "pod-b"
    # the same lease 31 s later: expired, taken over, released after the step (which then fails at the provider switch)
    out = host.task_step({"op": "process", "task": _task(), "now": 1021.5, "podName": "pod-a",
                          "objects": cluster + _objs(("Lease", lease("pod-b", 990.0)))})
    assert "unsupported provider: cohere" in out["task"]["status"]["error"] and "lease" not in out
    # our own lease: re-acquired at once
    out = host.task_step({"op": "process", "task": _task(), "now": 1000.0, "podName": "pod-a",
                          "objects": cluster + _objs(("Lease", lease("pod-a", 999.0)))})
    assert "unsupported provider: cohere" in out["task"]["status"]["error"]
    # lease skipped (INTEGRATION.md §5): two API writes fewer per step, a foreign lease is not even read
    with_lease = host.task_step(dict(base))
    assert with_lease["store_writes"] == 4
    out = host.task_step({"op": "process", "task": _task(), "emulate_lease": False, "now": 1000.0, "podName": "pod-a",
                          "objects": cluster + _objs(("Lease", lease("pod-b", 999.0)))})
    assert "unsupported provider: cohere" in out["task"]["status"]["error"]


def test_splitk_rule_and_workspace():
    """The engine's split-K rule (csrc/model_config.cc, pure host logic).  (1) Steps of <= 256 rows: the factor is a
    function of (M, K) only — batch invariance.  (2) Steps of more than 256 rows: the fewest fp32 planes whose wave
    count is within 15 % of the best (64 tiles -> 2, 96 -> 3, 128 -> 1), none once every SM has a tile.  (3) The
    workspace holds the planes of EVERY step height up to max_batch — a B = 1024 Mixtral step (O-proj: 128 tiles,
    formerly 8 planes against a workspace sized for 7 x 1024 rows) once overflowed it and stopped the engine."""
    import ctypes
    from agentcontrolplane_b200 import _lib
    lib = _lib.load_host()
    f = lib.acp_host_splitk_factor
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_int] * 5
    w = lib.acp_host_splitk_workspace_bytes
    w.restype = ctypes.c_size_t
    w.argtypes = [ctypes.c_int] * 5
    shapes = {"qkv": (6144, 4096), "o": (4096, 4096), "gate_up": (28672, 4096), "down": (4096, 14336),
              "70b_o_shard": (8192, 1024), "mixtral_qkv_shard": (768, 4096), "mixtral_o_shard": (4096, 512)}
    for name, (M, K) in shapes.items():
        small = {f(M, K, n, 222, 0) for n in (1, 7, 64, 200, 256)}
        assert len(small) == 1, (name, small)                      # (1)
        assert {f(M, K, n, 222, 1) for n in (300, 512, 1024)} == small, name   # strict mode keeps them everywhere
    assert (f(6144, 4096, 64, 222, 0), f(4096, 4096, 64, 222, 0), f(28672, 4096, 64, 222, 0), f(4096, 14336, 64, 222, 0)) == (5, 7, 1, 7)
    # (2) B = 512 at Llama-3-8B (config 2): 96 / 64 / 448 / 64 tiles
    assert (f(6144, 4096, 512, 222, 0), f(4096, 4096, 512, 222, 0), f(28672, 4096, 512, 222, 0), f(4096, 14336, 512, 222, 0)) == (3, 2, 1, 2)
    assert f(4096, 4096, 1024, 222, 0) == 1                        # 128 tiles: one plane, not eight
    assert f(4096, 4096, 2048, 222, 0) == 1                        # >= 148 tiles: never split
    # (3) every step height fits the workspace, for every shape and both modes
    for name, (M, K) in shapes.items():
        for strict in (0, 1):
            for max_batch in (64, 256, 512, 1000, 1024, 2048):
                ws = w(M, K, max_batch, 222, strict)
                for n in range(1, max_batch + 1, 7):
                    assert f(M, K, n, 222, strict) * n * M * 4 <= ws, (name, strict, max_batch, n)
                assert f(M, K, max_batch, 222, strict) * max_batch * M * 4 <= ws
