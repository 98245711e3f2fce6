// host/hostsim.cc — C entry points of include/acp_host.h: test hooks over the host mirror, the
// loopback stub completion server and the reconcile-loop simulator used by bench.py.
#include "acp_host.h"
#include <arpa/inet.h>
#include <netinet/in.h>
#include <netinet/tcp.h>
#include <string.h>
#include <sys/socket.h>
#include <unistd.h>
#include <algorithm>
#include <atomic>
#include <cmath>
#include <functional>
#include <map>
#include <mutex>
#include <set>
#include <condition_variable>
#include <chrono>
#include <thread>
#include "../chat.h"
#include "../model_config.h"
#include "../safetensors.h"
#include "task.h"

using namespace acp;
using acp::llmclient::Message;
using acp::llmclient::Tool;

static char* dup_out(const std::string& s, size_t* len = nullptr) {
  char* p = (char*)malloc(s.size() + 1);
  if (!p) return nullptr;
  memcpy(p, s.data(), s.size());
  p[s.size()] = 0;
  if (len) *len = s.size();
  return p;
}
extern "C" void acp_host_free(void* p) { free(p); }

static int ret_json(const Json& j, char** out) {
  *out = dup_out(j.dump());
  return *out ? ACP_OK : ACP_ERR_NOMEM;
}

static bool tools_from_json(const Json& arr, std::vector<Tool>* tools) {
  for (const Json& t : arr.items()) {
    Tool tool;
    tool.Type = t.get("type").as_string();
    if (tool.Type.empty()) tool.Type = "function";
    const Json& fn = t.get("function");
    tool.Function.Name = fn.get("name").as_string();
    tool.Function.Description = fn.get("description").as_string();
    tool.Function.Parameters = fn.get("parameters");
    tool.ACPToolType = t.get("acpToolType").as_string();
    tools->push_back(std::move(tool));
  }
  return true;
}

// ---------------------------------------------------------------------------------
// mock client: llmmocks.NewMockLLMClient in the reference's tests
// ---------------------------------------------------------------------------------
namespace {
class MockClient : public llmclient::LLMClient {
 public:
  explicit MockClient(const Json& spec, std::string* request_sink) : spec_(spec), sink_(request_sink) {}
  bool SendRequest(const llmclient::Context&, const std::vector<Message>& messages,
                   const std::vector<Tool>& tools, Message* out, llmclient::Error* err) override {
    if (sink_) *sink_ = llmclient::build_chat_request_json("mock", messages, tools, 0, nullptr);
    if (spec_.find("error")) { err->Message = spec_.get("error").as_string(); return false; }
    if (spec_.find("request_error")) {
      err->is_request_error = true;
      err->StatusCode = (int)spec_.get("request_error").get("status").as_int(400);
      err->Message = spec_.get("request_error").get("message").as_string();
      return false;
    }
    llmclient::message_from_crd_json(spec_.get("message"), out);
    return true;
  }

 private:
  Json spec_;
  std::string* sink_;
};
}  // namespace

// ---------------------------------------------------------------------------------
// stub completion server
// ---------------------------------------------------------------------------------
namespace {
struct StubServer {
  int listen_fd = -1;
  int port = 0;
  std::string body;
  std::atomic<bool> stop{false};
  std::thread thread;
  std::atomic<long long> served{0};
  // connection handlers are detached threads: stop() shuts their sockets down and waits for the
  // last one to leave before the server object is freed (found by the ThreadSanitizer build)
  std::mutex conn_mu;
  std::condition_variable conn_cv;
  std::set<int> conn_fds;
};
StubServer* g_stubs[16] = {nullptr};
std::mutex g_stub_mu;

void serve_conn_loop(StubServer* s, int fd);
void serve_conn(StubServer* s, int fd) {
  serve_conn_loop(s, fd);
  std::lock_guard<std::mutex> lk(s->conn_mu);
  s->conn_fds.erase(fd);
  close(fd);
  s->conn_cv.notify_all();
}

void serve_conn_loop(StubServer* s, int fd) {
  // HTTP/1.1 keep-alive: serve requests on this connection until the peer closes it
  std::string buf_acc;
  char buf[16384];
  while (true) {
    size_t he;
    while ((he = buf_acc.find("\r\n\r\n")) == std::string::npos) {
      ssize_t n = recv(fd, buf, sizeof buf, 0);
      if (n <= 0) return;
      buf_acc.append(buf, (size_t)n);
    }
    size_t cl = buf_acc.find("Content-Length:");
    const size_t len = (cl == std::string::npos || cl > he) ? 0 : (size_t)atoll(buf_acc.c_str() + cl + 15);
    const size_t need = he + 4 + len;
    while (buf_acc.size() < need) {
      ssize_t n = recv(fd, buf, sizeof buf, 0);
      if (n <= 0) return;
      buf_acc.append(buf, (size_t)n);
    }
    buf_acc.erase(0, need);
    const std::string resp = "HTTP/1.1 200 OK\r\nContent-Type: application/json\r\nContent-Length: " +
                             std::to_string(s->body.size()) + "\r\n\r\n" + s->body;
    size_t off = 0;
    while (off < resp.size()) {
      ssize_t n = send(fd, resp.data() + off, resp.size() - off, MSG_NOSIGNAL);
      if (n <= 0) return;
      off += (size_t)n;
    }
    ++s->served;
  }
}

void stub_loop(StubServer* s) {
  while (!s->stop) {
    sockaddr_in peer;
    socklen_t pl = sizeof peer;
    int fd = accept(s->listen_fd, (sockaddr*)&peer, &pl);
    if (fd < 0) { if (s->stop) break; continue; }
    int one = 1;
    setsockopt(fd, IPPROTO_TCP, TCP_NODELAY, &one, sizeof one);
    {
      std::lock_guard<std::mutex> lk(s->conn_mu);
      s->conn_fds.insert(fd);
    }
    std::thread(serve_conn, s, fd).detach();  // one goroutine per connection, like net/http
  }
}
}  // namespace

extern "C" int acp_host_stub_server_start(const char* body, int* port) {
  if (!port) return ACP_ERR_INVALID;
  StubServer* s = new StubServer();
  s->body = body ? body : "{\"id\":\"test-id\",\"choices\":[{\"message\":{\"content\":\"test\"}}]}";
  s->listen_fd = socket(AF_INET, SOCK_STREAM, 0);
  int one = 1;
  setsockopt(s->listen_fd, SOL_SOCKET, SO_REUSEADDR, &one, sizeof one);
  sockaddr_in addr;
  memset(&addr, 0, sizeof addr);
  addr.sin_family = AF_INET;
  addr.sin_addr.s_addr = htonl(INADDR_LOOPBACK);
  addr.sin_port = 0;
  if (bind(s->listen_fd, (sockaddr*)&addr, sizeof addr) != 0 || listen(s->listen_fd, 1024) != 0) {
    close(s->listen_fd);
    delete s;
    return ACP_ERR_INVALID;
  }
  socklen_t al = sizeof addr;
  getsockname(s->listen_fd, (sockaddr*)&addr, &al);
  s->port = ntohs(addr.sin_port);
  *port = s->port;
  s->thread = std::thread(stub_loop, s);
  std::lock_guard<std::mutex> lk(g_stub_mu);
  for (int i = 0; i < 16; ++i)
    if (!g_stubs[i]) { g_stubs[i] = s; return i; }
  return ACP_ERR_NOMEM;
}

extern "C" void acp_host_stub_server_stop(int handle) {
  StubServer* s = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_stub_mu);
    if (handle < 0 || handle >= 16 || !g_stubs[handle]) return;
    s = g_stubs[handle];
    g_stubs[handle] = nullptr;
  }
  s->stop = true;
  shutdown(s->listen_fd, SHUT_RDWR);
  close(s->listen_fd);
  if (s->thread.joinable()) s->thread.join();
  {
    std::unique_lock<std::mutex> lk(s->conn_mu);
    for (int fd : s->conn_fds) shutdown(fd, SHUT_RDWR);   // wakes handlers blocked in recv on keep-alive sockets
    s->conn_cv.wait(lk, [&] { return s->conn_fds.empty(); });
  }
  delete s;
}

// ---------------------------------------------------------------------------------
// chat-side hooks
// ---------------------------------------------------------------------------------
namespace {
// tokenizer.json files loaded for the test hooks, by path (nullptr / "" / "synthetic" = built in)
const Tokenizer* hook_tokenizer(const char* path, std::string* err) {
  if (!path || !*path || std::string(path) == "synthetic") return &synthetic_tokenizer();
  static std::mutex mu;
  static std::map<std::string, std::unique_ptr<Tokenizer>> cache;
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(path);
  if (it != cache.end()) return it->second.get();
  std::unique_ptr<Tokenizer> t = load_tokenizer_json(path, err);
  if (!t) return nullptr;
  return (cache[path] = std::move(t)).get();
}
int tokenizer_error(const std::string& err, char** out_json) {
  Json j = Json::object();
  j.set("error", Json(err));
  ret_json(j, out_json);
  return ACP_ERR_INVALID;
}
}  // namespace

extern "C" int acp_host_tokenizer_encode(const char* tokenizer_path, const char* text, size_t len, char** out_json) {
  if (!text || !out_json) return ACP_ERR_INVALID;
  std::string err;
  const Tokenizer* tok = hook_tokenizer(tokenizer_path, &err);
  if (!tok) return tokenizer_error(err, out_json);
  const std::string s(text, len);
  std::vector<int> ids;
  tok->encode(s, &ids);
  std::vector<std::string> pieces;
  llama3_pretokenize(s, &pieces);
  Json out = Json::object(), a = Json::array(), p = Json::array();
  for (int t : ids) a.push(Json(t));
  for (const std::string& x : pieces) p.push(Json(x));
  out.set("ids", a);
  out.set("pieces", p);
  out.set("kind", Json(tok->kind()));
  out.set("vocab_size", Json(tok->vocab_size()));
  Json sp = Json::object();
  sp.set("begin_of_text", Json(tok->special().begin_of_text)); sp.set("end_of_text", Json(tok->special().end_of_text));
  sp.set("start_header", Json(tok->special().start_header)); sp.set("end_header", Json(tok->special().end_header));
  sp.set("eom", Json(tok->special().eom)); sp.set("eot", Json(tok->special().eot));
  sp.set("python_tag", Json(tok->special().python_tag));
  out.set("special", sp);
  return ret_json(out, out_json);
}

extern "C" int acp_host_tokenizer_decode(const char* tokenizer_path, const int* ids, int n, char** out_text, size_t* out_len) {
  if ((!ids && n > 0) || !out_text) return ACP_ERR_INVALID;
  std::string err;
  const Tokenizer* tok = hook_tokenizer(tokenizer_path, &err);
  if (!tok) return ACP_ERR_INVALID;
  std::vector<int> v(ids, ids + n);
  *out_text = dup_out(tok->decode(v), out_len);
  return *out_text ? ACP_OK : ACP_ERR_NOMEM;
}

extern "C" int acp_host_render_prompt_with(const char* tokenizer_path, const char* chat_request_json, size_t len,
                                           char** out_json) {
  if (!chat_request_json || !out_json) return ACP_ERR_INVALID;
  std::string err;
  const Tokenizer* tok = hook_tokenizer(tokenizer_path, &err);
  if (!tok) return tokenizer_error(err, out_json);
  ChatRequest req;
  Json out = Json::object();
  int status = parse_chat_request(chat_request_json, len, &req, &err);
  if (status != 0) {
    out.set("status", Json(status));
    out.set("error", Json(err));
    return ret_json(out, out_json);
  }
  std::vector<int> ids;
  render_prompt(req, &ids, *tok);
  Json arr = Json::array();
  for (int t : ids) arr.push(Json(t));
  out.set("text", Json(render_prompt_text(req)));
  out.set("token_ids", arr);
  return ret_json(out, out_json);
}

extern "C" int acp_host_render_prompt(const char* chat_request_json, size_t len, char** out_json) {
  if (!chat_request_json || !out_json) return ACP_ERR_INVALID;
  ChatRequest req;
  std::string err;
  Json out = Json::object();
  int status = parse_chat_request(chat_request_json, len, &req, &err);
  if (status != 0) {
    out.set("status", Json(status));
    out.set("error", Json(err));
    return ret_json(out, out_json);
  }
  std::vector<int> ids;
  if (req.has_prompt_ids) ids = req.prompt_token_ids; else render_prompt(req, &ids);
  Json arr = Json::array();
  for (int t : ids) arr.push(Json(t));
  out.set("text", Json(render_prompt_text(req)));
  out.set("token_ids", arr);
  return ret_json(out, out_json);
}

extern "C" int acp_host_parse_completion(const char* text, size_t len, const char* tools_json,
                                         const char* call_id_prefix, char** out_json) {
  if (!text || !out_json) return ACP_ERR_INVALID;
  std::vector<ToolDef> tools;
  if (tools_json && *tools_json) {
    Json arr;
    std::string err;
    if (!Json::parse(std::string(tools_json), &arr, &err)) return ACP_ERR_INVALID;
    for (const Json& t : arr.items()) {
      ToolDef td;
      td.type = "function";
      td.name = t.get("function").get("name").as_string();
      tools.push_back(td);
    }
  }
  ParsedCompletion pc = parse_completion(std::string(text, len), tools, call_id_prefix ? call_id_prefix : "call_");
  Json out = Json::object();
  if (!pc.tool_calls.empty()) {
    Json tcs = Json::array();
    for (auto& t : pc.tool_calls) {
      Json fn = Json::object();
      fn.set("name", Json(t.name));
      fn.set("arguments", Json(t.arguments));
      Json o = Json::object();
      o.set("id", Json(t.id));
      o.set("type", Json(t.type));
      o.set("function", fn);
      tcs.push(o);
    }
    out.set("tool_calls", tcs);
  } else {
    out.set("content", Json(pc.content));
  }
  return ret_json(out, out_json);
}

extern "C" int acp_host_decode_tokens(const int* ids, int n, char** out_text, size_t* out_len) {
  if ((!ids && n > 0) || !out_text) return ACP_ERR_INVALID;
  std::vector<int> v(ids, ids + n);
  *out_text = dup_out(decode_tokens(v), out_len);
  return *out_text ? ACP_OK : ACP_ERR_NOMEM;
}

extern "C" int acp_host_build_chat_request(const char* model, const char* messages_crd_json,
                                           const char* tools_json, char** out_json) {
  if (!messages_crd_json || !out_json) return ACP_ERR_INVALID;
  Json msgs, tools;
  std::string err;
  if (!Json::parse(std::string(messages_crd_json), &msgs, &err)) return ACP_ERR_INVALID;
  if (tools_json && *tools_json && !Json::parse(std::string(tools_json), &tools, &err)) return ACP_ERR_INVALID;
  std::vector<Message> mv;
  for (const Json& m : msgs.items()) { Message mm; llmclient::message_from_crd_json(m, &mm); mv.push_back(mm); }
  std::vector<Tool> tv;
  tools_from_json(tools, &tv);
  *out_json = dup_out(llmclient::build_chat_request_json(model ? model : "", mv, tv, 0, nullptr));
  return *out_json ? ACP_OK : ACP_ERR_NOMEM;
}

extern "C" int acp_host_convert_response(const char* response_json, char** out_message_crd_json) {
  if (!response_json || !out_message_crd_json) return ACP_ERR_INVALID;
  Message m;
  std::string err;
  if (!llmclient::convert_from_response_json(response_json, &m, &err)) return ACP_ERR_INVALID;
  return ret_json(llmclient::message_to_crd_json(m), out_message_crd_json);
}

// ---------------------------------------------------------------------------------
// one state-machine operation
// ---------------------------------------------------------------------------------
static Json result_json(const task::Result& r) {
  Json j = Json::object();
  j.set("requeue", Json(r.Requeue));
  j.set("requeueAfter", Json(r.RequeueAfter));
  return j;
}

extern "C" int acp_host_task_step(acp_engine* engine, const char* input_json, char** out_json) {
  if (!input_json || !out_json) return ACP_ERR_INVALID;
  Json in;
  std::string perr;
  if (!Json::parse(std::string(input_json), &in, &perr)) return ACP_ERR_INVALID;
  task::ObjectStore store;
  task::Recorder rec;
  task::StateMachine sm(&store, &rec);
  task::Task t;
  if (!task::task_from_json(in.get("task"), &t)) return ACP_ERR_INVALID;
  std::vector<Tool> tools;
  tools_from_json(in.get("tools"), &tools);
  for (const Json& tcj : in.get("toolcalls").items())
    store.Put("ToolCall", tcj.get("metadata").get("name").as_string(), tcj);
  long long writes0 = store.writes();
  const std::string op = in.get("op").as_string();
  std::string err, request_json;
  task::Result res;
  // cluster objects the step may look up: [{"kind": "Agent"|"LLM"|"Secret"|"ContactChannel", "object": {...}}]
  for (const Json& o : in.get("objects").items())
    store.Put(o.get("kind").as_string(), o.get("object").get("metadata").get("name").as_string(), o.get("object"));
  writes0 = store.writes();   // API writes of the step itself, not of the fixture
  if (op == "checkToolCalls") {
    res = sm.checkToolCalls(&t, &err);
  } else if (op == "sendLLMRequestFromCluster") {
    // the whole ReadyForLLM arm: validateTaskAndAgent, getLLMAndCredentials, CreateClient, collectTools, LLM step
    task::MCPToolsByServer mcp;
    for (const auto& kv : in.get("mcp").members()) mcp[kv.first] = kv.second.items();
    store.Put("Task", t.Name, task::task_to_json(t));
    writes0 = store.writes();
    llmclient::Context ctx;
    res = sm.sendLLMRequestFromCluster(ctx, &t, mcp, engine, &err);
  } else if (op == "process" || op == "reconcile") {
    // StateMachine.Process / TaskReconciler.Reconcile against the objects given; "now" pins the lease clock,
    // "podName" this controller's identity, "emulate_lease": false = the local provider's hand-off
    task::MCPToolsByServer mcp;
    for (const auto& kv : in.get("mcp").members()) mcp[kv.first] = kv.second.items();
    if (in.find("now")) { const double fixed = in.get("now").as_double(); sm.now = [fixed] { return fixed; }; }
    if (in.find("podName")) sm.podName = in.get("podName").as_string();
    if (in.find("emulate_lease")) sm.emulate_lease = in.get("emulate_lease").as_bool(true);
    llmclient::Context ctx;
    if (op == "process") {
      if (!in.get("unsaved").as_bool(false)) { store.Put("Task", t.Name, task::task_to_json(t)); writes0 = store.writes(); }
      res = sm.Process(ctx, &t, mcp, engine, &err);
    } else {
      // Reconcile fetches the Task itself: it only exists if it is among "objects"
      Json tj;
      task::TaskReconciler rec2(&store, &rec);
      if (in.find("now")) { const double fixed = in.get("now").as_double(); rec2.stateMachine().now = [fixed] { return fixed; }; }
      res = rec2.Reconcile(ctx, in.get("name").as_string(), mcp, engine, &err);
      if (store.Get("Task", in.get("name").as_string(), &tj)) task::task_from_json(tj, &t);
    }
    Json lease;
    if (store.Get("Lease", "task-llm-" + t.Name, &lease)) { /* reported below */ }
  } else if (op == "collectTools") {
    task::MCPToolsByServer mcp;
    for (const auto& kv : in.get("mcp").members()) mcp[kv.first] = kv.second.items();
    tools = sm.collectTools(in.get("agent"), mcp);
  } else {
    const Json& llm = in.get("llm");
    const std::string provider = llm.get("provider").as_string();
    llmclient::BaseConfig bc;
    bc.Model = llm.get("model").as_string();
    bc.BaseURL = llm.get("baseURL").as_string();
    bc.MaxTokens = (int)llm.get("maxTokens").as_int(0);
    task::ClientFactory factory = [&](std::string* cerr) -> std::unique_ptr<llmclient::LLMClient> {
      if (provider == "mock")
        return std::unique_ptr<llmclient::LLMClient>(new MockClient(llm.get("mock"), &request_json));
      auto c = llmclient::NewLLMClient(provider, "test-key", bc, engine, cerr);
      if (c && provider == "local" && llm.get("acp").is_object())
        static_cast<llmclient::LocalClient*>(c.get())->set_extension(llm.get("acp"));
      return c;
    };
    llmclient::Context ctx;
    res = sm.sendLLMRequest(ctx, &t, tools, factory, &err);
  }
  Json out = Json::object();
  out.set("task", task::task_to_json(t));
  out.set("result", result_json(res));
  out.set("error", Json(err));
  Json evs = Json::array();
  for (auto& e : rec.events) {
    Json ej = Json::object();
    ej.set("type", Json(e.Type));
    ej.set("reason", Json(e.Reason));
    ej.set("message", Json(e.Message));
    evs.push(ej);
  }
  out.set("events", evs);
  Json tcs = Json::array();
  if (!t.Status.ToolCallRequestID.empty())
    for (Json& j : store.ListToolCalls(t.Name, t.Status.ToolCallRequestID)) tcs.push(j);
  out.set("toolcalls", tcs);
  out.set("store_writes", Json(store.writes() - writes0));
  {
    Json lease;
    if (store.Get("Lease", "task-llm-" + t.Name, &lease)) out.set("lease", lease);
  }
  if (op == "collectTools") {
    Json tj = Json::array();
    for (const Tool& tl : tools) {
      Json o = Json::object(), fn = Json::object();
      fn.set("name", Json(tl.Function.Name));
      fn.set("description", Json(tl.Function.Description));
      fn.set("parameters", tl.Function.Parameters);
      o.set("type", Json(tl.Type));
      o.set("function", fn);
      o.set("acpToolType", Json(tl.ACPToolType));
      tj.push(o);
    }
    out.set("tools", tj);
  }
  if (!request_json.empty()) out.set("request_json", Json(request_json));
  return ret_json(out, out_json);
}

// ---------------------------------------------------------------------------------
// reconcile-loop simulator
// ---------------------------------------------------------------------------------
static uint64_t mix64(uint64_t z) {
  z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27; z *= 0x94D049BB133111EBull;
  z ^= z >> 31;
  return z;
}

// user content of `n` ASCII letters/spaces, deterministic in (seed, task)
static std::string synth_text(uint64_t seed, int task, int n) {
  std::string s;
  s.reserve(n);
  static const char alphabet[] = "abcdefghijklmnopqrstuvwxyz    ";
  for (int i = 0; i < n; ++i)
    s.push_back(alphabet[mix64(seed * 1000003ull + (uint64_t)task * 7919ull + (uint64_t)i) % 30]);
  return s;
}

extern "C" int acp_host_splitk_factor(int M, int K, int N, int target_ctas, int strict) {
  return acp::splitk_factor(M, K, N, target_ctas, strict != 0);
}
extern "C" size_t acp_host_splitk_workspace_bytes(int M, int K, int max_batch, int target_ctas, int strict) {
  return acp::splitk_workspace_bytes(M, K, max_batch, target_ctas, strict != 0);
}

extern "C" int acp_host_checkpoint_index(const char* path, char** out_json) {
  if (!path || !out_json) return ACP_ERR_INVALID;
  acp::Checkpoint ck;
  std::string err;
  auto fail = [&](const std::string& e) {
    Json j = Json::object();
    j.set("error", Json(e));
    ret_json(j, out_json);
    return ACP_ERR_INVALID;
  };
  if (!ck.open(path, &err)) return fail(err);
  Json out;
  std::string perr;
  if (!Json::parse(ck.index_json(), &out, &perr)) return fail(perr);
  if (!ck.has_config()) return fail("no config.json in " + ck.dir());
  acp::ModelConfig mc;
  if (!acp::model_config_from_hf(ck.config(), &mc, &err)) return fail(err);
  Json m = Json::object();
  m.set("hidden", Json(mc.hidden)); m.set("layers", Json(mc.layers)); m.set("heads", Json(mc.heads));
  m.set("kv_heads", Json(mc.kv_heads)); m.set("ffn", Json(mc.ffn)); m.set("vocab", Json(mc.vocab));
  m.set("rope_theta", Json(mc.rope_theta)); m.set("eps", Json((double)mc.eps));
  m.set("tied_embeddings", Json(mc.tied_embeddings)); m.set("max_pos", Json(mc.max_pos));
  float inv[64];
  acp::rope_inv_freq(mc, inv);
  Json fr = Json::array();
  for (float f : inv) fr.push(Json((double)f));
  m.set("rope_inv_freq", fr);
  out.set("model", m);
  return ret_json(out, out_json);
}

extern "C" int acp_host_checkpoint_tensor_bf16(const char* path, const char* name, uint16_t* out, size_t max_elems,
                                               size_t* n_elems) {
  if (!path || !name || !n_elems) return ACP_ERR_INVALID;
  acp::Checkpoint ck;
  std::string err;
  if (!ck.open(path, &err)) return ACP_ERR_INVALID;
  const acp::StTensor* t = ck.find(name);
  if (!t) return ACP_ERR_NOT_FOUND;
  *n_elems = (size_t)t->numel();
  if (!out) return ACP_OK;
  if (max_elems < *n_elems) return ACP_ERR_INVALID;
  return acp::st_to_bf16(*t, 0, *n_elems, out) ? ACP_OK : ACP_ERR_INVALID;
}

// completion the calling worker's next LLM step is forced to emit ("" = free-running); namespace scope: a
// function-local thread_local is only initialised in threads that execute its declaration
static thread_local std::string tl_script;

extern "C" int acp_hostsim_run(acp_engine* engine, const char* config_json, char** result_json_out) {
  if (!config_json || !result_json_out) return ACP_ERR_INVALID;
  Json cfg;
  std::string perr;
  if (!Json::parse(std::string(config_json), &cfg, &perr) || !cfg.is_object()) return ACP_ERR_INVALID;
  const int n_tasks = (int)cfg.get("tasks").as_int(1);
  const int workers = std::max(1, (int)cfg.get("workers").as_int(1));
  const std::string provider = cfg.get("provider").as_string().empty() ? "local" : cfg.get("provider").as_string();
  llmclient::BaseConfig bc;
  bc.Model = cfg.get("model").as_string();
  bc.BaseURL = cfg.get("baseURL").as_string();
  bc.MaxTokens = (int)cfg.get("max_tokens").as_int(64);
  const int prompt_tokens = (int)cfg.get("prompt_tokens").as_int(0);
  // BASELINE config 2: window lengths log-uniform on [prompt_tokens_min, prompt_tokens_max] (seeded per Task)
  const int pt_min = (int)cfg.get("prompt_tokens_min").as_int(0), pt_max = (int)cfg.get("prompt_tokens_max").as_int(0);
  const bool mixed = pt_min > 0 && pt_max >= pt_min;
  const int n_tools = (int)cfg.get("tools").as_int(0);
  const bool tool_loop = cfg.get("tool_loop").as_bool(false);
  // BASELINE config 4: open-loop Poisson arrivals (Tasks/s, seeded exponential gaps; 0 = all at once) and
  // sub-agent delegation chains of this depth (root -> sub-agent-1 -> ... ; executor.go:176-242)
  const double arrival_rate = cfg.get("arrival_rate").as_double(0.0);
  const int delegation_depth = std::max(0, std::min(4, (int)cfg.get("delegation_depth").as_int(0)));
  const uint64_t seed = (uint64_t)cfg.get("seed").as_int(1);
  const bool lease = cfg.find("emulate_lease") ? cfg.get("emulate_lease").as_bool(true) : true;
  // report status.output of every root Task (by index) in the result: what the Task's owner reads back
  const bool return_outputs = cfg.get("return_outputs").as_bool(false);
  if (provider == "local" && !engine) return ACP_ERR_INVALID;

  // agent-level tool list (collectTools): synthetic MCP tools server__tool_i
  std::vector<Json> mcp;
  for (int i = 0; i < n_tools; ++i) {
    Json t = Json::object();
    t.set("name", Json("tool_" + std::to_string(i)));
    t.set("description", Json("synthetic tool " + std::to_string(i)));
    Json url = Json::object(); url.set("type", Json("string"));
    Json props = Json::object(); props.set("url", url);
    Json schema = Json::object();
    schema.set("type", Json("object"));
    schema.set("properties", props);
    t.set("inputSchema", schema);
    mcp.push_back(t);
  }
  const std::vector<Tool> tools = task::ConvertMCPTools(mcp, "fetch");

  task::ObjectStore store;
  task::Recorder rec;
  const std::string system_prompt = "You are a helpful test assistant.";  // test_getting_started.go:279
  // size the user message so that the rendered window is exactly prompt_tokens tokens
  auto render_len = [&](const std::string& user) {
    ChatRequest cr;
    ChatMessage s; s.role = "system"; s.content = system_prompt;
    ChatMessage u; u.role = "user"; u.content = user;
    cr.messages = {s, u};
    for (const Tool& t : tools) {
      ToolDef td; td.type = t.Type; td.name = t.Function.Name; td.description = t.Function.Description;
      td.parameters = t.Function.Parameters;
      cr.tools.push_back(td);
    }
    std::vector<int> ids;
    render_prompt(cr, &ids);
    return (int)ids.size();
  };
  const int overhead = render_len("");
  int user_len = 30;  // "What is the capital of France?" scale when no target is given
  int window_tokens = 0;
  if (prompt_tokens > 0) {
    // the synthetic tokenizer is byte-level below id 256, so an agent's tool schemas alone can
    // exceed a small target: the window is then "overhead + a short user message" and the
    // result reports the real length (bench.py sizes its KV pool from it)
    user_len = std::max(16, prompt_tokens - overhead);
    window_tokens = overhead + user_len;
  }
  long long window_sum = 0;
  int window_max = 0;
  const bool dry_run = cfg.get("dry_run").as_bool(false);   // sizes only: no Task is reconciled
  for (int i = 0; i < n_tasks; ++i) {
    int this_user_len = user_len;
    if (mixed) {
      // length = exp(U(ln min, ln max)), U from the splitmix of (length seed, task index); the length
      // seed is fixed per configuration ("length_seed") so that every step runs the same distribution
      const uint64_t ls = (uint64_t)cfg.get("length_seed").as_int(0xC0F162);
      const double u = (double)(mix64(ls * 0x9E3779B97F4A7C15ull + (uint64_t)i) >> 11) / 9007199254740992.0;
      const int target = (int)std::exp(std::log((double)pt_min) + u * (std::log((double)pt_max) - std::log((double)pt_min)));
      this_user_len = std::max(16, target - overhead);
    }
    window_sum += overhead + this_user_len;
    window_max = std::max(window_max, overhead + this_user_len);
    if (dry_run) continue;
    task::Task t;
    t.Name = "task-" + std::to_string(i);
    t.UID = "uid-" + std::to_string(i);
    t.AgentName = "test-agent";
    t.Status.Phase = "ReadyForLLM";
    t.Status.Status = "Ready";
    t.Status.ContextWindow = task::buildInitialContextWindow(
        {}, system_prompt, (prompt_tokens > 0 || mixed) ? synth_text(seed, i, this_user_len) : std::string("What is the capital of France?"));
    store.Put("Task", t.Name, task::task_to_json(t));
  }

  // the cluster objects the reference's sendLLMRequest looks up on every step (validateTaskAndAgent,
  // getLLMAndCredentials, collectTools): one Agent, its LLM, the API-key Secret
  {
    Json agent = Json::object(), ameta = Json::object(), aspec = Json::object(), astatus = Json::object();
    ameta.set("name", Json("test-agent"));
    Json llmref = Json::object(); llmref.set("name", Json("test-llm"));
    aspec.set("llmRef", llmref);
    aspec.set("system", Json(system_prompt));
    if (n_tools > 0) {
      Json srv = Json::object(); srv.set("name", Json("fetch"));
      Json servers = Json::array(); servers.push(srv);
      aspec.set("mcpServers", servers);
    }
    astatus.set("ready", Json(true));
    if (delegation_depth > 0) {
      Json ref = Json::object(); ref.set("name", Json("sub-agent-1"));
      Json subs = Json::array(); subs.push(ref);
      aspec.set("subAgents", subs);
    }
    agent.set("metadata", ameta); agent.set("spec", aspec); agent.set("status", astatus);
    store.Put("Agent", "test-agent", agent);
    for (int d = 1; d <= delegation_depth; ++d) {   // sub-agent-d delegates to sub-agent-(d+1); the last one answers
      Json sa = Json::object(), sm_ = Json::object(), ss = Json::object(), st = Json::object();
      sm_.set("name", Json("sub-agent-" + std::to_string(d)));
      ss.set("llmRef", llmref);
      ss.set("system", Json("You are sub-agent " + std::to_string(d) + "."));
      ss.set("description", Json("delegate level " + std::to_string(d)));
      if (d < delegation_depth) {
        Json ref = Json::object(); ref.set("name", Json("sub-agent-" + std::to_string(d + 1)));
        Json subs = Json::array(); subs.push(ref);
        ss.set("subAgents", subs);
      }
      st.set("ready", Json(true));
      sa.set("metadata", sm_); sa.set("spec", ss); sa.set("status", st);
      store.Put("Agent", "sub-agent-" + std::to_string(d), sa);
    }
    Json llm = Json::object(), lmeta = Json::object(), lspec = Json::object(), params = Json::object();
    lmeta.set("name", Json("test-llm"));
    lspec.set("provider", Json(provider));
    params.set("model", Json(bc.Model));
    if (!bc.BaseURL.empty()) params.set("baseUrl", Json(bc.BaseURL));
    if (bc.MaxTokens > 0) params.set("maxTokens", Json(bc.MaxTokens));
    lspec.set("parameters", params);
    if (provider != "local") {   // `local` needs no credentials (INTEGRATION.md §4)
      Json ref = Json::object(); ref.set("name", Json("test-secret")); ref.set("key", Json("api-key"));
      Json from = Json::object(); from.set("secretKeyRef", ref);
      lspec.set("apiKeyFrom", from);
      Json secret = Json::object(), smeta = Json::object(), data = Json::object();
      smeta.set("name", Json("test-secret"));
      data.set("api-key", Json("test-key"));
      secret.set("metadata", smeta); secret.set("data", data);
      store.Put("Secret", "test-secret", secret);
    }
    llm.set("metadata", lmeta); llm.set("spec", lspec);
    store.Put("LLM", "test-llm", llm);
  }
  task::MCPToolsByServer mcp_by_server;
  if (n_tools > 0) mcp_by_server["fetch"] = mcp;
  const std::string scripted_call = tools.empty() ? std::string()
      : "{\"name\": \"" + tools[0].Function.Name + "\", \"parameters\": {\"url\": \"https://api.example.com/data\"}}";

  std::atomic<int> next{0};
  std::atomic<long long> reconciles{0};
  std::mutex lat_mu;
  std::vector<double> lat_ms;
  std::map<std::string, int> phases;
  std::string first_error;
  uint64_t digest = 0;
  // ONE state machine shared by all reconcile workers, like the reference's TaskReconciler
  task::StateMachine sm(&store, &rec);
  sm.emulate_lease = lease;
  sm.client_hook = [&](llmclient::LLMClient* c) {
    if (tl_script.empty()) return;
    // scripted step: force the model's output to be a tool call (BASELINE configs 3 and 4).  The call must
    // fit the completion budget or it is cut mid-JSON (one token per byte under the synthetic vocabulary):
    // never fewer decode steps than configured.
    auto* lc = static_cast<llmclient::LocalClient*>(c);
    if (bc.MaxTokens < (int)tl_script.size() + 1) lc->set_max_tokens((int)tl_script.size() + 1);
    Json ext = Json::object();
    Json forced = Json::array();
    for (unsigned char ch : tl_script) forced.push(Json((int)ch));
    forced.push(Json(TOK_EOT));
    ext.set("force_tokens", forced);
    lc->set_extension(ext);
  };
  // arrival offsets of the root Tasks (seconds from the start of the run)
  std::vector<double> arrival((size_t)std::max(0, n_tasks), 0.0);
  if (arrival_rate > 0.0) {
    double tcur = 0.0;
    for (int i = 0; i < n_tasks; ++i) {
      const double u = ((double)(mix64(seed * 0xA24BAED4963EE407ull + (uint64_t)i) >> 11) + 0.5) / 9007199254740992.0;
      tcur += -std::log(u) / arrival_rate;
      arrival[(size_t)i] = tcur;
    }
  }
  std::vector<double> task_ms;   // arrival -> terminal phase of every ROOT Task
  std::vector<std::string> outputs(return_outputs ? (size_t)std::max(0, n_tasks) : 0);
  const auto t0 = std::chrono::steady_clock::now();
  // Runs one Task (root or delegated child) to a terminal phase on the calling worker: the Task controller's
  // reconciles, with the (out of scope) ToolCall controller emulated in between — plain tools "execute" at once
  // with a fixed result; a delegate_to_agent__X ToolCall creates the child Task like executeDelegateToAgent
  // (toolcall/executor.go:176-242), the child runs to its end, and its Output becomes the ToolCall's Result
  // (waitForSubAgent, toolcall/state_machine.go:218-267).
  std::function<void(const std::string&, int, int)> run_task = [&](const std::string& name, int index, int level) {
    int steps = 0;
    for (int guard = 0; guard < 24; ++guard) {
      Json tj;
      if (!store.Get("Task", name, &tj)) return;  // r.getTask (task_controller.go:216)
      task::Task t;
      task::task_from_json(tj, &t);
      const std::string& phase = t.Status.Phase;
      llmclient::Context ctx;
      std::string err;
      if (phase.empty() || phase == "Initializing" || phase == "Pending") {
        sm.Process(ctx, &t, mcp_by_server, engine, &err);   // initialize / validateAgent (delegated children start here)
        if (!err.empty()) return;
      } else if (phase == "ReadyForLLM") {
        const auto s0 = std::chrono::steady_clock::now();
        tl_script.clear();
        if (provider == "local" && steps == 0) {
          if (level < delegation_depth)
            tl_script = "{\"name\": \"delegate_to_agent__sub-agent-" + std::to_string(level + 1) + "\", \"parameters\": {\"message\": \"" +
                        synth_text(seed ^ 0xD1E6, index * 8 + level, 96) + "\"}}";
          else if (tool_loop && !tools.empty() && level == 0)
            tl_script = scripted_call;
        }
        sm.Process(ctx, &t, mcp_by_server, engine, &err);   // -> sendLLMRequest (a5, a6, CreateClient, a8, the LLM step)
        tl_script.clear();
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - s0).count();
        ++reconciles;
        {
          std::lock_guard<std::mutex> lk(lat_mu);
          lat_ms.push_back(ms);
        }
        ++steps;
        if (!err.empty()) {        // would requeue after 5 s; out of the timed loop
          std::lock_guard<std::mutex> lk(lat_mu);
          if (first_error.empty()) first_error = name + " (phase " + t.Status.Phase + "): " + err;
          return;
        }
      } else if (phase == "ToolCallsPending") {
        for (Json& tcj : store.ListToolCalls(name, t.Status.ToolCallRequestID)) {
          task::ToolCall tc;
          task::toolcall_from_json(tcj, &tc);
          if (tc.ToolType == "DelegateToAgent") {
            const std::string agentName = tc.ToolRef.substr(std::min(tc.ToolRef.size(), std::string("delegate_to_agent__").size()));
            Json args;
            std::string perr2;
            if (!Json::parse(tc.Arguments, &args, &perr2) || !args.get("message").is_string()) {
              tc.StatusStatus = "Error";
              tc.StatusResult = "missing or invalid 'message' argument";
            } else {
              std::string child = "delegate-" + tc.Name + "-" + agentName;
              if (child.size() > 63) child = child.substr(0, 55) + "-" + child.substr(child.size() - 7);
              task::Task ct;
              ct.Name = child;
              ct.UID = "uid-" + child;
              ct.AgentName = agentName;
              ct.UserMessage = args.get("message").as_string();
              ct.Labels["acp.humanlayer.dev/parent-toolcall"] = tc.Name;
              store.Create("Task", child, task::task_to_json(ct));
              run_task(child, index, level + 1);
              Json cj;
              task::Task done;
              if (store.Get("Task", child, &cj)) task::task_from_json(cj, &done);
              if (done.Status.Phase == "FinalAnswer") { tc.StatusStatus = "Succeeded"; tc.StatusResult = done.Status.Output; }
              else { tc.StatusStatus = "Error"; tc.StatusResult = done.Status.Error.empty() ? "Sub-agent task failed" : done.Status.Error; }
            }
          } else {
            tc.StatusStatus = "Succeeded";
            tc.StatusResult = "{\"data\": \"" + synth_text(seed ^ 0x5151, index, 96) + "\"}";
          }
          store.Put("ToolCall", tc.Name, task::toolcall_to_json(tc));
        }
        sm.Process(ctx, &t, mcp_by_server, engine, &err);   // -> checkToolCalls
      } else {
        return;  // FinalAnswer / Failed
      }
    }
  };
  auto worker = [&]() {
    while (true) {
      const int i = next.fetch_add(1);
      if (i >= n_tasks) break;
      const std::string name = "task-" + std::to_string(i);
      if (arrival_rate > 0.0)
        std::this_thread::sleep_until(t0 + std::chrono::duration_cast<std::chrono::steady_clock::duration>(
                                               std::chrono::duration<double>(arrival[(size_t)i])));
      const auto a0 = std::chrono::steady_clock::now();
      run_task(name, i, 0);
      const double total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a0).count();
      Json tj;
      if (store.Get("Task", name, &tj)) {
        task::Task t;
        task::task_from_json(tj, &t);
        std::lock_guard<std::mutex> lk(lat_mu);
        task_ms.push_back(total_ms);
        ++phases[t.Status.Phase];
        if (return_outputs) outputs[(size_t)i] = t.Status.Output;
        if (t.Status.Phase == "Failed" && first_error.empty())
          first_error = name + ": " + (t.Status.Error.empty() ? t.Status.StatusDetail : t.Status.Error);
        uint64_t h = 1469598103934665603ull;
        const std::string d = t.Status.Output + "|" + t.Status.Phase;
        for (unsigned char ch : d) { h ^= ch; h *= 1099511628211ull; }
        digest ^= mix64(h + (uint64_t)i);
      }
    }
  };
  std::vector<std::thread> pool;
  for (int w = 0; w < workers && !dry_run; ++w) pool.emplace_back(worker);
  for (auto& th : pool) th.join();
  const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();

  std::sort(lat_ms.begin(), lat_ms.end());
  Json out = Json::object();
  out.set("reconciles", Json((long long)reconciles.load()));
  out.set("tasks", Json(n_tasks));
  out.set("workers", Json(workers));
  out.set("wall_s", Json(wall));
  out.set("reconciles_per_s", Json(wall > 0 ? reconciles.load() / wall : 0.0));
  if (!lat_ms.empty()) {
    out.set("step_ms_p50", Json(lat_ms[lat_ms.size() / 2]));
    out.set("step_ms_p99", Json(lat_ms[std::min(lat_ms.size() - 1, (size_t)(lat_ms.size() * 0.99))]));
  }
  if (!task_ms.empty()) {
    std::sort(task_ms.begin(), task_ms.end());
    out.set("task_ms_p50", Json(task_ms[task_ms.size() / 2]));
    out.set("task_ms_p99", Json(task_ms[std::min(task_ms.size() - 1, (size_t)(task_ms.size() * 0.99))]));
  }
  out.set("store_writes", Json(store.writes()));
  out.set("store_reads", Json(store.reads()));
  out.set("prompt_tokens", Json(prompt_tokens > 0 ? window_tokens : overhead + user_len));
  out.set("prompt_tokens_total", Json(window_sum));
  out.set("prompt_tokens_max", Json(window_max));
  Json ph = Json::object();
  for (auto& kv : phases) ph.set(kv.first, Json(kv.second));
  out.set("final_phases", ph);
  if (!first_error.empty()) out.set("first_error", Json(first_error));   // why the first Failed Task failed
  if (return_outputs) {
    Json arr = Json::array();
    for (const std::string& o : outputs) arr.push(Json(o));
    out.set("outputs", arr);
  }
  char dbuf[32];
  snprintf(dbuf, sizeof dbuf, "%016llx", (unsigned long long)digest);
  out.set("digest", Json(std::string(dbuf)));
  return ret_json(out, result_json_out);
}
